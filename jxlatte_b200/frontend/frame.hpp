// frame.hpp -- one frame: TOC, LFGlobal, LF groups (LF coefficients, HF metadata), HFGlobal (quant-table parameters,
// coefficient orders), pass groups (HF coefficient decode, modular group streams).  Output = the post-entropy frame
// state jxlb200_vardct_reconstruct() takes, stitched to frame level, plus the frame-level modular channels and their
// transform list.  Follows jxlatte: J/frame/Frame.java:129-200,271-462, LFGlobal.java, group/LFGroup.java, group/Pass.java,
// group/PassGroup.java:67-84, vardct/LFCoefficients.java, HFMetadata.java, HFBlockContext.java, HFGlobal.java:194-302,
// HFPass.java, HFCoefficients.java:49-138,230-265.
#pragma once
#include <array>
#include <cmath>
#include <map>

#include "headers.hpp"
#include "modular.hpp"

namespace jxlf {

struct TType { int param_index, order_id, method, ph, pw; };
inline const TType kTypes[27] = {
    {0, 0, 0, 8, 8},      {1, 1, 3, 8, 8},      {2, 1, 1, 8, 8},     {3, 1, 2, 8, 8},      {4, 2, 0, 16, 16},    {5, 3, 0, 32, 32},   {6, 4, 0, 16, 8},
    {6, 4, 0, 8, 16},     {7, 5, 0, 32, 8},     {7, 5, 0, 8, 32},    {8, 6, 0, 32, 16},    {8, 6, 0, 16, 32},    {9, 1, 5, 8, 8},     {9, 1, 4, 8, 8},
    {10, 1, 6, 8, 8},     {10, 1, 6, 8, 8},     {10, 1, 6, 8, 8},    {10, 1, 6, 8, 8},     {11, 7, 0, 64, 64},   {12, 8, 0, 64, 32},  {12, 8, 0, 32, 64},
    {13, 9, 0, 128, 128}, {14, 10, 0, 128, 64}, {14, 10, 0, 64, 128}, {15, 11, 0, 256, 256}, {16, 12, 0, 256, 128}, {16, 12, 0, 128, 256}};
inline bool type_flips(int t) { return kTypes[t].ph > kTypes[t].pw || (kTypes[t].method == 0 && kTypes[t].ph == kTypes[t].pw); }
// the non-vertical shape of each coefficient order / quant-table parameter set: (rows, cols) in pixels
inline const int kOrderShape[13][2] = {{8, 8}, {8, 8}, {16, 16}, {32, 32}, {8, 16}, {8, 32}, {16, 32}, {64, 64}, {32, 64}, {128, 128}, {64, 128}, {256, 256}, {128, 256}};
inline const int kParamShape[17][2] = {{8, 8}, {8, 8}, {8, 8}, {8, 8}, {16, 16}, {32, 32}, {8, 16}, {8, 32}, {16, 32}, {8, 8}, {8, 8},
                                        {64, 64}, {32, 64}, {128, 128}, {64, 128}, {256, 256}, {128, 256}};

// mirrors jxlb200_qm_params (include/jxlb200.h) minus the raw pointers
struct QuantParams {
    int mode = 0, n_dct = 0, n_param = 0, n_4x4 = 0;
    float denominator = 0.0f;
    float dct_param[3][17] = {{0}}, param[3][9] = {{0}}, params4x4[3][17] = {{0}};
    std::vector<float> raw[3];
};

// Patch.readPatch (J/frame/features/Patch.java:18-60): pos = (x, y) per position; blend = (mode, alpha channel, clamp) per position
// and per channel group (colour, then each extra channel)
struct PatchInfo { int ref = 0, x0 = 0, y0 = 0, w = 0, h = 0; std::vector<int32_t> pos; std::vector<int32_t> blend; };

struct FrameData {
    FrameHeader hdr;
    int padded_w = 0, padded_h = 0;            // Frame.getPaddedFrameSize
    int num_groups = 0, num_lf_groups = 0, group_cols = 0, lf_group_cols = 0;
    uint64_t toc_bit_offset = 0, toc_first_section = 0;      // where the TOC starts (bits) and where the first section starts (bytes), in the codestream
    std::vector<uint32_t> toc_lengths;
    // LFGlobal
    float lf_dequant[3] = {1.0f / 4096, 1.0f / 512, 1.0f / 256};
    int global_scale = 0, quant_lf = 0;
    int color_factor = 84, x_factor_lf = 128, b_factor_lf = 128;
    float base_corr_x = 0.0f, base_corr_b = 1.0f;
    float noise[8] = {0};
    int num_patches = 0, num_splines = 0;
    std::vector<PatchInfo> patches;
    // SplinesBundle (J/frame/features/spline/SplinesBundle.java:25-75): control points (x, y) and 4 x 32 coefficients per spline
    struct SplineInfo { std::vector<int32_t> points; int32_t coeff[4][32]; };
    std::vector<SplineInfo> splines;
    int32_t spline_quant_adjust = 0;
    // VarDCT state, frame level
    std::vector<int32_t> qcoeff[3];
    std::vector<float> lf[3];
    std::vector<int32_t> lf_quant[3];            // the same planes before LFCoefficients' arithmetic (X, Y, B order), for the device LF kernel
    std::vector<uint8_t> lf_extra_precision;     // per LF group
    float scaled_dequant[3] = {0, 0, 0};
    std::vector<uint8_t> dct_select, block_origin;
    std::vector<int32_t> hf_mul, sharpness, x_from_y, b_from_y;
    bool quant_all_default = true;
    QuantParams qparams[17];
    // frame-level modular stream
    ModularStream modular;
    bool has_modular = false;
    bool lf_only = false;                        // parsed up to the LF groups only (JXLF_LF_ONLY): no HF state was read
};

class FrameDecoder {
  public:
    FrameDecoder(BitReader &br, const ImageHeader &ih) : br_(br), ih_(ih) {}

    // header + TOC; afterwards frame_bytes() is known, so a caller can skip the frame
    void read_header(FrameData &f) {
        br_.align();
        f.hdr.read(br_, ih_);
        const FrameHeader &h = f.hdr;
        // crop sizes are 30-bit fields: bound what a header may make this process allocate (2^28 px = the 16384^2 config)
        if (h.width <= 0 || h.height <= 0) throw StreamError("empty frame");
        if ((int64_t)h.width * h.height > (1ll << 28) || h.width > (1 << 24) || h.height > (1 << 24))
            throw Unsupported("frame larger than 2^28 pixels");
        f.group_cols = ceil_div(h.width, h.group_dim);
        f.lf_group_cols = ceil_div(h.width, h.group_dim << 3);
        f.num_groups = f.group_cols * ceil_div(h.height, h.group_dim);
        f.num_lf_groups = f.lf_group_cols * ceil_div(h.height, h.group_dim << 3);
        const int fy = 1 << std::max(h.shift_y[0], std::max(h.shift_y[1], h.shift_y[2]));
        const int fx = 1 << std::max(h.shift_x[0], std::max(h.shift_x[1], h.shift_x[2]));
        if (h.encoding == ENC_VARDCT) {
            f.padded_h = (ceil_div((h.height + 7) >> 3, fy) * fy) << 3;
            f.padded_w = (ceil_div((h.width + 7) >> 3, fx) * fx) << 3;
        } else {
            f.padded_h = ceil_div(h.height, fy) * fy;
            f.padded_w = ceil_div(h.width, fx) * fx;
        }
        if (f.hdr.num_passes > 1) coverage().multi_pass_frames++;
        read_toc(f);
    }
    size_t frame_bytes() const { size_t n = 0; for (auto l : toc_len_) n += l; return n; }
    void skip(FrameData &) { br_.seek_bytes(toc_start_ + frame_bytes()); }

    // lf_only: stop after LfGlobal and the LF groups' LF coefficients and Modular channels.  HF metadata, HfGlobal and the pass
    // groups are never read, so their sections may hold anything.
    void decode(FrameData &f, bool lf_only = false) {
        f.lf_only = lf_only;
        open_sections();
        fc_.group_dim = f.hdr.group_dim;
        fc_.modular_h = f.hdr.height;
        fc_.modular_w = f.hdr.width;
        fc_.bit_depth = ih_.depth.bits;
        fc_.ec_dim_shift.clear();
        for (auto &e : ih_.extra) fc_.ec_dim_shift.push_back(e.dim_shift);
        read_lf_global(f, section(0));
        allocate_vardct(f);
        decode_lf_groups(f);
        if (!lf_only) {
            BitReader &hg = section(1 + f.num_lf_groups);
            if (f.hdr.encoding == ENC_VARDCT) read_hf_global(f, hg);
            read_passes(f, hg);
            decode_pass_groups(f);
        }
        br_.seek_bytes(toc_start_ + frame_bytes());
    }

  private:
    BitReader &br_;
    const ImageHeader &ih_;
    FrameContext fc_;
    MATree global_tree_;
    std::vector<uint32_t> toc_len_, toc_perm_;
    size_t toc_start_ = 0;
    std::vector<BitReader> sections_;
    // HFBlockContext
    std::vector<uint8_t> block_ctx_map_;
    int num_block_clusters_ = 15, num_lf_contexts_ = 1;
    std::vector<int32_t> lf_thresholds_[3];
    std::vector<int32_t> qf_thresholds_;
    float scaled_dequant_[3] = {0, 0, 0};
    // per LF group, kept for the HF pass
    struct LFGroupState {
        int bh = 0, bw = 0;                      // size in 8x8 blocks
        std::vector<int32_t> lf_index;           // bh * bw
        std::vector<uint8_t> dct_select;         // 255 = free
        std::vector<int32_t> hf_mul;
        std::vector<uint32_t> blocks;            // (y << 16) | x in placement order
    };
    std::vector<LFGroupState> lfg_;
    int num_hf_presets_ = 1;
    struct PassState {
        int min_shift = 0, max_shift = 3;
        std::vector<int> replaced;               // indices into the global channel list
        std::vector<uint32_t> order[13][3];      // (y << 16) | x, natural order when not coded
        EntropyStream coeff_stream;
    };
    std::vector<PassState> passes_;

    // ---- TOC (Frame.java:152-186) and permutations (:206-226) ----
    static std::vector<uint32_t> read_permutation(BitReader &br, EntropyStream &es, uint32_t size, uint32_t skip) {
        auto ctx = [](uint32_t x) { return std::min(7, ceil_log1p(x)); };
        const uint32_t end = es.read(br, ctx(size));
        if (end > size - skip) throw StreamError("permutation: illegal end value");
        std::vector<uint32_t> lehmer(size, 0);
        for (uint32_t i = skip; i < end + skip; i++) {
            lehmer[i] = es.read(br, ctx(i > skip ? lehmer[i - 1] : 0));
            if (lehmer[i] >= size - i) throw StreamError("permutation: illegal Lehmer code");
        }
        std::vector<uint32_t> pool(size), perm(size);
        for (uint32_t i = 0; i < size; i++) pool[i] = i;
        const uint32_t coded = end + skip;          // Lehmer digits beyond this are zero: the rest of the pool follows in order
        for (uint32_t i = 0; i < coded; i++) {
            perm[i] = pool[lehmer[i]];
            pool.erase(pool.begin() + lehmer[i]);
        }
        std::copy(pool.begin(), pool.end(), perm.begin() + coded);
        return perm;
    }
    void read_toc(FrameData &f) {
        f.toc_bit_offset = br_.position();
        const size_t entries = (f.num_groups == 1 && f.hdr.num_passes == 1) ? 1 : 2 + f.num_lf_groups + (size_t)f.num_groups * f.hdr.num_passes;
        toc_perm_.clear();
        if (br_.flag()) {
            coverage().permuted_toc++;
            EntropyStream es(br_, 8);
            toc_perm_ = read_permutation(br_, es, (uint32_t)entries, 0);
            es.expect_final_state("TOC permutation");
        }
        br_.align();
        toc_len_.resize(entries);
        for (auto &l : toc_len_) l = br_.u32(0, 10, 1024, 14, 17408, 22, 4211712, 30);
        br_.align();
        toc_start_ = (size_t)(br_.position() >> 3);
        f.toc_first_section = toc_start_;
        f.toc_lengths.assign(toc_len_.begin(), toc_len_.end());
    }
    void open_sections() {
        sections_.clear();
        size_t at = toc_start_;
        std::vector<BitReader> physical;
        for (auto l : toc_len_) {
            if (at + l > br_.size()) throw StreamError("TOC entry runs past the end of the stream");
            physical.emplace_back(br_.data() + at, l);
            at += l;
        }
        sections_.resize(physical.size());
        for (size_t i = 0; i < physical.size(); i++) sections_[i] = physical[toc_perm_.empty() ? i : toc_perm_[i]];
    }
    BitReader &section(size_t logical) { return sections_.size() <= 1 ? sections_[0] : sections_.at(logical); }

    // ---- LFGlobal ----
    void read_lf_global(FrameData &f, BitReader &br) {
        const FrameHeader &h = f.hdr;
        const int extra = (int)ih_.extra.size();
        if (h.flags & FLAG_PATCHES) {
            int alpha_channels = 0;
            for (auto &e : ih_.extra) alpha_channels += e.type == 0;
            EntropyStream es(br, 10);
            f.num_patches = (int)es.read(br, 0);
            // a one-symbol ANS distribution costs no bits per symbol, so the counts are untrusted: bound patches and positions by
            // the frame's pixel count (a patch position names at least one pixel), capped like the spline control points
            const uint64_t patch_cap = std::min<uint64_t>((uint64_t)std::max(h.width, 1) * (uint64_t)std::max(h.height, 1), 1u << 20);
            if (f.num_patches < 0 || (uint64_t)f.num_patches > patch_cap) throw StreamError("too many patches");
            uint64_t total_positions = 0;
            f.patches.resize(f.num_patches);
            for (PatchInfo &pt : f.patches) {
                pt.ref = (int)es.read(br, 1);
                pt.x0 = (int)es.read(br, 3);
                pt.y0 = (int)es.read(br, 3);
                pt.w = 1 + (int)es.read(br, 2);
                pt.h = 1 + (int)es.read(br, 2);
                const uint32_t count = 1 + es.read(br, 7);
                if ((int32_t)count <= 0) throw StreamError("patch count overflow");
                total_positions += count;
                if (total_positions > patch_cap) throw StreamError("too many patch positions");
                int32_t px = 0, py = 0;
                for (uint32_t j = 0; j < count; j++) {
                    if (j == 0) {
                        px = (int32_t)es.read(br, 4);
                        py = (int32_t)es.read(br, 4);
                    } else {
                        const int32_t dx = unpack_signed(es.read(br, 6)), dy = unpack_signed(es.read(br, 6));
                        px = detail::wrap_add(dx, px);
                        py = detail::wrap_add(dy, py);
                    }
                    pt.pos.push_back(px);
                    pt.pos.push_back(py);
                    for (int k = 0; k < extra + 1; k++) {
                        const uint32_t mode = es.read(br, 5);
                        if (mode >= 8) throw StreamError("illegal patch blend mode");
                        int32_t alpha = 0, clamp = 0;
                        if (mode > 3 && alpha_channels > 1) {
                            alpha = (int32_t)es.read(br, 8);
                            if (alpha >= extra) throw StreamError("patch alpha channel out of range");
                        }
                        if (mode > 2) clamp = es.read(br, 9) != 0;
                        pt.blend.push_back((int32_t)mode);
                        pt.blend.push_back(alpha);
                        pt.blend.push_back(clamp);
                    }
                }
            }
            es.expect_final_state("patches");
        }
        if (h.flags & FLAG_SPLINES) {
            if (ih_.color_channels() < 3) throw StreamError("splines in a greyscale image");
            EntropyStream es(br, 6);
            f.num_splines = 1 + (int)es.read(br, 2);
            f.splines.resize(f.num_splines);
            std::vector<int32_t> start(2 * (size_t)f.num_splines);
            for (int i = 0; i < f.num_splines; i++) {
                int32_t x = (int32_t)es.read(br, 1), y = (int32_t)es.read(br, 1);
                if (i) {
                    x = detail::wrap_add(unpack_signed((uint32_t)x), start[2 * i - 2]);
                    y = detail::wrap_add(unpack_signed((uint32_t)y), start[2 * i - 1]);
                }
                start[2 * i] = x;
                start[2 * i + 1] = y;
            }
            f.spline_quant_adjust = unpack_signed(es.read(br, 0));
            for (int i = 0; i < f.num_splines; i++) {
                FrameData::SplineInfo &sp = f.splines[i];
                const uint32_t points = 1 + es.read(br, 3);
                if (points > (1u << 20)) throw StreamError("too many spline control points");
                std::vector<int32_t> dx(points - 1), dy(points - 1);
                for (uint32_t j = 0; j + 1 < points; j++) {
                    dx[j] = unpack_signed(es.read(br, 4));
                    dy[j] = unpack_signed(es.read(br, 4));
                }
                int32_t cx = start[2 * i], cy = start[2 * i + 1], ddx = 0, ddy = 0;
                sp.points = {cx, cy};
                for (uint32_t j = 1; j < points; j++) {
                    ddy = detail::wrap_add(ddy, dy[j - 1]);
                    ddx = detail::wrap_add(ddx, dx[j - 1]);
                    cy = detail::wrap_add(cy, ddy);
                    cx = detail::wrap_add(cx, ddx);
                    sp.points.push_back(cx);
                    sp.points.push_back(cy);
                }
                for (int k = 0; k < 4; k++)                      // X, Y, B, sigma
                    for (int j = 0; j < 32; j++) sp.coeff[k][j] = unpack_signed(es.read(br, 5));
            }
            es.expect_final_state("splines");
        }
        if (h.flags & FLAG_NOISE) {
            if (ih_.color_channels() < 3) throw StreamError("noise in a greyscale image");
            for (float &v : f.noise) v = (float)br.bits(10) / 1024.0f;
        }
        if (!br.flag())
            for (float &v : f.lf_dequant) v = br.f16() * (1.0f / 128.0f);
        if (h.encoding == ENC_VARDCT) {
            f.global_scale = (int)br.u32(1, 11, 2049, 11, 4097, 12, 8193, 16);
            f.quant_lf = (int)br.u32(16, 0, 1, 5, 1, 8, 1, 16);
            for (int i = 0; i < 3; i++) scaled_dequant_[i] = (float)(1 << 16) * f.lf_dequant[i] / (float)(f.global_scale * f.quant_lf);
            for (int i = 0; i < 3; i++) f.scaled_dequant[i] = scaled_dequant_[i];
            read_block_context(br);
            if (!br.flag()) {
                f.color_factor = (int)br.u32(84, 0, 256, 0, 2, 8, 258, 16);
                f.base_corr_x = br.f16();
                f.base_corr_b = br.f16();
                f.x_factor_lf = (int)br.bits(8);
                f.b_factor_lf = (int)br.bits(8);
            }
        }
        if (br.flag()) {
            global_tree_ = MATree();
            global_tree_.read(br);
            fc_.global_tree = &global_tree_;
        } else {
            fc_.global_tree = nullptr;
        }
        int ec_start = 0;
        if (h.encoding == ENC_MODULAR) ec_start = (!h.do_ycbcr && !ih_.xyb_encoded && ih_.color.color_space == 1) ? 1 : 3;
        f.modular.init_global(br, fc_, 0, extra + ec_start, ec_start);
        f.has_modular = extra + ec_start > 0;
        f.modular.decode_channels(br, true);
    }

    void read_block_context(BitReader &br) {                 // HFBlockContext.java:22-57
        for (auto &t : lf_thresholds_) t.clear();
        qf_thresholds_.clear();
        if (br.flag()) {
            static const uint8_t kDefault[39] = {0, 1, 2, 2, 3, 3, 4, 5, 6, 6, 6, 6, 6, 7, 8, 9, 9, 10, 11, 12, 13, 14, 14, 14, 14, 14,
                                                 7, 8, 9, 9, 10, 11, 12, 13, 14, 14, 14, 14, 14};
            block_ctx_map_.assign(kDefault, kDefault + 39);
            num_block_clusters_ = 15;
            num_lf_contexts_ = 1;
            return;
        }
        coverage().custom_block_ctx++;
        int lf_ctx = 1, size = 39;
        for (auto &t : lf_thresholds_) {
            t.resize(br.bits(4));
            lf_ctx *= (int)t.size() + 1;
            for (auto &v : t) v = unpack_signed(br.u32(0, 4, 16, 8, 272, 16, 65808, 32));
        }
        num_lf_contexts_ = lf_ctx;
        qf_thresholds_.resize(br.bits(4));
        for (auto &v : qf_thresholds_) v = 1 + (int32_t)br.u32(0, 2, 4, 3, 12, 5, 44, 8);
        size *= (int)qf_thresholds_.size() + 1;
        size *= lf_ctx;
        if (size > 39 * 64) throw StreamError("HF block context map too large");
        num_block_clusters_ = EntropyStream::read_cluster_map(br, block_ctx_map_, size, 16);
    }

    void allocate_vardct(FrameData &f) {
        if (f.hdr.encoding != ENC_VARDCT) return;
        const int bh = f.padded_h >> 3, bw = f.padded_w >> 3;
        for (int c = 0; c < 3; c++) {
            f.lf[c].assign((size_t)(bh >> f.hdr.shift_y[c]) * (bw >> f.hdr.shift_x[c]), 0.0f);
            f.lf_quant[c].assign((size_t)(bh >> f.hdr.shift_y[c]) * (bw >> f.hdr.shift_x[c]), 0);
        }
        if (f.lf_only) return;
        for (int c = 0; c < 3; c++) f.qcoeff[c].assign((size_t)(f.padded_h >> f.hdr.shift_y[c]) * (f.padded_w >> f.hdr.shift_x[c]), 0);
        f.dct_select.assign((size_t)bh * bw, 0);
        f.block_origin.assign((size_t)bh * bw, 0);
        f.hf_mul.assign((size_t)bh * bw, 1);
        f.sharpness.assign((size_t)bh * bw, 0);
        const int th = (f.padded_h + 63) >> 6, tw = (f.padded_w + 63) >> 6;
        f.x_from_y.assign((size_t)th * tw, 0);
        f.b_from_y.assign((size_t)th * tw, 0);
    }

    // channels of the frame-level modular stream that a group-level stream fills in, cut to the group's rectangle
    std::vector<Channel> cut_channels(const FrameData &f, const std::vector<int> &which, int group, int dim) {
        std::vector<Channel> out;
        for (int idx : which) {
            Channel c = f.modular.channels[idx];
            c.px.clear();
            c.decoded = false;
            if (c.vshift < 0 || c.vshift > 30 || c.hshift < 0 || c.hshift > 30) throw StreamError("modular channel shift out of range");
            const int gh = dim >> c.vshift, gw = dim >> c.hshift;
            if (gh <= 0 || gw <= 0) throw StreamError("modular channel shift exceeds the group size");
            const int stride = ceil_div(c.w, gw);
            c.oy = (group / std::max(stride, 1)) * gh;
            c.ox = (group % std::max(stride, 1)) * gw;
            c.h = std::max(0, std::min(c.h - c.oy, gh));
            c.w = std::max(0, std::min(c.w - c.ox, gw));
            out.push_back(std::move(c));
        }
        return out;
    }
    static void paste_channels(FrameData &f, const std::vector<int> &which, const ModularStream &ms) {
        if (ms.channels.size() < which.size()) throw StreamError("group modular stream lost channels");
        for (size_t j = 0; j < which.size(); j++) {
            Channel &dst = f.modular.channels[which[j]];
            const Channel &src = ms.channels[j];
            dst.allocate();
            for (int y = 0; y < src.h; y++) {
                if (src.oy + y >= dst.h) break;
                const int n = std::min(src.w, dst.w - src.ox);
                if (n > 0) std::memcpy(&dst.at(src.oy + y, src.ox), &src.px[(size_t)y * src.w], sizeof(int32_t) * n);
            }
        }
    }

    // ---- LF groups (Frame.java:271-308, LFGroup.java) ----
    void decode_lf_groups(FrameData &f) {
        const FrameHeader &h = f.hdr;
        std::vector<int> lf_channels;
        for (size_t i = 0; i < f.modular.channels.size(); i++) {
            const Channel &c = f.modular.channels[i];
            if (!c.decoded && c.vshift >= 3 && c.hshift >= 3) lf_channels.push_back((int)i);
        }
        lfg_.assign(f.num_lf_groups, LFGroupState());
        const int lf_dim = h.group_dim << 3;
        for (int idx : lf_channels) f.modular.channels[idx].allocate();
        // LF groups are independent sections writing disjoint rectangles: one task each (the reference decodes them one
        // after the other on the caller's thread)
        parallel_sections(f.num_lf_groups, [&](int g) {
            BitReader &br = section(1 + g);
            const int gy = g / f.lf_group_cols, gx = g % f.lf_group_cols;
            LFGroupState &st = lfg_[g];
            st.bh = std::min(lf_dim, f.padded_h - gy * lf_dim) >> 3;
            st.bw = std::min(lf_dim, f.padded_w - gx * lf_dim) >> 3;
            if (h.encoding == ENC_VARDCT) read_lf_coefficients(f, br, g, st);
            ModularStream ms;
            ms.init(br, fc_, 1 + f.num_lf_groups + g, cut_channels(f, lf_channels, g, lf_dim));
            ms.decode_channels(br);
            paste_channels(f, lf_channels, ms);
            if (h.encoding == ENC_VARDCT && !f.lf_only) read_hf_metadata(f, br, g, st);
        });
    }

    // Runs body(0..n-1); in parallel when the frame has one TOC section per task (a single-section frame shares one reader).
    // The first exception is re-thrown on the calling thread, invalid-stream errors before anything else.
    template <class Body> void parallel_sections(int n, Body body) {
        if (sections_.size() <= 1 || n <= 1) {
            for (int i = 0; i < n; i++) body(i);
            return;
        }
        std::string stream_err, unsupported_err, other_err;
#pragma omp parallel for schedule(dynamic, 1)
        for (int i = 0; i < n; i++) {
            try {
                body(i);
            } catch (const Unsupported &e) {
#pragma omp critical(jxlf_err)
                if (unsupported_err.empty()) unsupported_err = e.what();
            } catch (const StreamError &e) {
#pragma omp critical(jxlf_err)
                if (stream_err.empty()) stream_err = e.what();
            } catch (const std::exception &e) {
#pragma omp critical(jxlf_err)
                if (other_err.empty()) other_err = e.what();
            }
        }
        if (!stream_err.empty()) throw StreamError(stream_err);
        if (!unsupported_err.empty()) throw Unsupported(unsupported_err);
        if (!other_err.empty()) throw std::runtime_error(other_err);
    }

    // LFCoefficients.java:20-98 (dequant, LF chroma-from-luma, adaptive smoothing) and :100-194
    void read_lf_coefficients(FrameData &f, BitReader &br, int g, LFGroupState &st) {
        const FrameHeader &h = f.hdr;
        if (h.flags & FLAG_USE_LF_FRAME) {
            // LFCoefficients.java:39-52: the LF planes are copied from the LF frame decoded earlier (the caller owns its pixels,
            // so f.lf stays zero here and is filled in by the caller); lfIndex stays all zero
            st.lf_index.assign((size_t)st.bh * st.bw, 0);
            return;
        }
        const bool subsampled = h.shift_y[0] | h.shift_y[1] | h.shift_y[2] | h.shift_x[0] | h.shift_x[1] | h.shift_x[2];
        const bool smooth = !(h.flags & FLAG_SKIP_ADAPTIVE_LF_SMOOTHING);
        if (smooth && subsampled) throw StreamError("adaptive LF smoothing with chroma subsampling");
        static const int kMap[3] = {1, 0, 2};               // component i lives in modular channel kMap[i] (Y, X, B order)
        std::vector<Channel> info(3);
        int ch_h[3], ch_w[3];
        for (int i = 0; i < 3; i++) {
            ch_h[i] = st.bh >> h.shift_y[i];
            ch_w[i] = st.bw >> h.shift_x[i];
            info[kMap[i]] = Channel(ch_h[i], ch_w[i], h.shift_y[i], h.shift_x[i]);
        }
        const int extra_precision = (int)br.bits(2);
        if (f.lf_extra_precision.size() != (size_t)f.num_lf_groups) f.lf_extra_precision.assign(f.num_lf_groups, 0);
        f.lf_extra_precision[g] = (uint8_t)extra_precision;
        ModularStream ms;
        ms.init(br, fc_, 1 + g, std::move(info));
        ms.decode_channels(br);
        if (ms.channels.size() != 3) throw StreamError("LF coefficient stream must end with three channels");
        std::vector<float> dq[3];
        for (int i = 0; i < 3; i++) {
            const Channel &q = ms.channels[kMap[i]];
            if (q.h != ch_h[i] || q.w != ch_w[i]) throw StreamError("LF coefficient channel changed shape");
            const float sd = scaled_dequant_[i] / (float)(1 << extra_precision);
            dq[i].resize(q.px.size());
            for (size_t k = 0; k < q.px.size(); k++) dq[i][k] = (float)q.px[k] * sd;
        }
        if (!subsampled) {
            const float kx = f.base_corr_x + ((float)f.x_factor_lf - 128.0f) / (float)f.color_factor;
            const float kb = f.base_corr_b + ((float)f.b_factor_lf - 128.0f) / (float)f.color_factor;
            for (size_t k = 0; k < dq[1].size(); k++) {
                dq[0][k] += kx * dq[1][k];
                dq[2][k] += kb * dq[1][k];
            }
        }
        if (smooth) { adaptive_smooth(dq, st.bh, st.bw); coverage().lf_smoothing++; }
        // stitch into the frame-level LF planes
        const int gy = g / f.lf_group_cols, gx = g % f.lf_group_cols;
        for (int i = 0; i < 3; i++) {
            const int fw = (f.padded_w >> 3) >> h.shift_x[i];
            const int y0 = (gy << 8) >> h.shift_y[i], x0 = (gx << 8) >> h.shift_x[i];
            const Channel &q = ms.channels[kMap[i]];
            for (int y = 0; y < ch_h[i]; y++) {
                std::memcpy(&f.lf[i][(size_t)(y0 + y) * fw + x0], &dq[i][(size_t)y * ch_w[i]], sizeof(float) * ch_w[i]);
                std::memcpy(&f.lf_quant[i][(size_t)(y0 + y) * fw + x0], &q.px[(size_t)y * ch_w[i]], sizeof(int32_t) * ch_w[i]);
            }
        }
        // LF context index per block (:183-202)
        st.lf_index.assign((size_t)st.bh * st.bw, 0);
        for (int y = 0; y < st.bh; y++)
            for (int x = 0; x < st.bw; x++) {
                int idx[3] = {0, 0, 0};
                for (int i = 0; i < 3; i++) {
                    const Channel &q = ms.channels[kMap[i]];
                    const int32_t v = q.at(y >> h.shift_y[i], x >> h.shift_x[i]);
                    for (int32_t t : lf_thresholds_[i]) idx[i] += v > t;
                }
                int li = idx[0];
                li = li * ((int)lf_thresholds_[2].size() + 1) + idx[2];
                li = li * ((int)lf_thresholds_[1].size() + 1) + idx[1];
                st.lf_index[(size_t)y * st.bw + x] = li;
            }
    }

    void adaptive_smooth(std::vector<float> (&co)[3], int h, int w) const {      // LFCoefficients.adaptiveSmooth :108-181
        if (h < 3 || w < 3) return;      // no interior sample: the reference leaves every value as it is
        std::vector<float> weighted[3], gap((size_t)h * w, 0.5f);
        for (int i = 0; i < 3; i++) {
            weighted[i].assign((size_t)h * w, 0.0f);
            const float sd = scaled_dequant_[i];
            const std::vector<float> &c = co[i];
            for (int y = 1; y < h - 1; y++)
                for (int x = 1; x < w - 1; x++) {
                    const size_t p = (size_t)y * w + x;
                    const float sample = c[p];
                    const float adjacent = c[p - 1] + c[p + 1] + c[p - w] + c[p + w];
                    const float diag = c[p - w - 1] + c[p - w + 1] + c[p + w - 1] + c[p + w + 1];
                    const float wv = 0.05226273532324128f * sample + 0.20345139757231578f * adjacent + 0.0334829185968739f * diag;
                    weighted[i][p] = wv;
                    const float gv = std::fabs(sample - wv) * sd;
                    if (gv > gap[p]) gap[p] = gv;
                }
        }
        for (float &gv : gap) gv = std::max(0.0f, 3.0f - 4.0f * gv);
        for (int i = 0; i < 3; i++)
            for (int y = 1; y < h - 1; y++)
                for (int x = 1; x < w - 1; x++) {
                    const size_t p = (size_t)y * w + x;
                    co[i][p] = (co[i][p] - weighted[i][p]) * gap[p] + weighted[i][p];
                }
    }

    // HFMetadata.java:22-57, placeBlock :93-119
    void read_hf_metadata(FrameData &f, BitReader &br, int g, LFGroupState &st) {
        const int nbits = ceil_log2((uint64_t)st.bh * st.bw);
        const int nb_blocks = 1 + (int)br.bits(nbits);
        const int th = (st.bh + 7) / 8, tw = (st.bw + 7) / 8;
        std::vector<Channel> info;
        info.emplace_back(th, tw, 0, 0);
        info.emplace_back(th, tw, 0, 0);
        info.emplace_back(2, nb_blocks, 0, 0);
        info.emplace_back(st.bh, st.bw, 0, 0);
        ModularStream ms;
        ms.init(br, fc_, 1 + 2 * f.num_lf_groups + g, std::move(info));
        ms.decode_channels(br);
        if (ms.channels.size() != 4) throw StreamError("HF metadata stream must end with four channels");
        const Channel &xfy = ms.channels[0], &bfy = ms.channels[1], &info2 = ms.channels[2], &sharp = ms.channels[3];
        if (info2.h != 2 || info2.w != nb_blocks || sharp.h != st.bh || sharp.w != st.bw || xfy.h != th || xfy.w != tw)
            throw StreamError("HF metadata channel changed shape");
        st.dct_select.assign((size_t)st.bh * st.bw, 255);
        st.hf_mul.assign((size_t)st.bh * st.bw, 0);
        st.blocks.clear();
        int ly = 0, lx = 0;
        for (int i = 0; i < nb_blocks; i++) {
            const int32_t type = info2.at(0, i);
            if (type < 0 || type > 26) throw StreamError("invalid transform type");
            const int bh = kTypes[type].ph >> 3, bw = kTypes[type].pw >> 3;
            const int32_t mul = detail::wrap_add(1, info2.at(1, i));
            bool placed = false;
            for (int y = ly, x = lx; y < st.bh && !placed; y++, x = 0) {
                for (; x < st.bw; x++) {
                    if (bw + x > st.bw) break;                       // too wide here: next row
                    bool occupied = false;
                    for (int ix = 0; ix < bw; ix++) {
                        const uint8_t t = st.dct_select[(size_t)y * st.bw + x + ix];
                        if (t != 255) {
                            x += (kTypes[t].pw >> 3) - 1;            // jxlatte skips by the width of the block it ran into
                            occupied = true;
                            break;
                        }
                    }
                    if (occupied) continue;
                    if (y + bh > st.bh) throw StreamError("varblock leaves the LF group");
                    for (int iy = 0; iy < bh; iy++)
                        for (int ix = 0; ix < bw; ix++) {
                            st.dct_select[(size_t)(y + iy) * st.bw + x + ix] = (uint8_t)type;
                            st.hf_mul[(size_t)(y + iy) * st.bw + x + ix] = mul;
                        }
                    st.blocks.push_back(((uint32_t)y << 16) | (uint32_t)x);
                    ly = y;
                    lx = x;
                    placed = true;
                    break;
                }
            }
            if (!placed) throw StreamError("could not find a place for a varblock");
        }
        // stitch to frame level
        const int gy = g / f.lf_group_cols, gx = g % f.lf_group_cols;
        const int fbw = f.padded_w >> 3, ftw = (f.padded_w + 63) >> 6;
        for (int y = 0; y < st.bh; y++)
            for (int x = 0; x < st.bw; x++) {
                const size_t src = (size_t)y * st.bw + x, dst = (size_t)((gy << 8) + y) * fbw + (gx << 8) + x;
                f.dct_select[dst] = st.dct_select[src] == 255 ? 0 : st.dct_select[src];
                f.hf_mul[dst] = st.dct_select[src] == 255 ? 1 : st.hf_mul[src];
                f.sharpness[dst] = sharp.at(y, x);
            }
        for (uint32_t b : st.blocks) f.block_origin[(size_t)((gy << 8) + (b >> 16)) * fbw + (gx << 8) + (b & 0xffff)] = 1;
        for (int y = 0; y < th; y++)
            for (int x = 0; x < tw; x++) {
                f.x_from_y[(size_t)((gy << 5) + y) * ftw + (gx << 5) + x] = xfy.at(y, x);
                f.b_from_y[(size_t)((gy << 5) + y) * ftw + (gx << 5) + x] = bfy.at(y, x);
            }
    }

    // ---- HFGlobal (HFGlobal.java:194-302): quant-table PARAMETERS; the tables themselves are built by jxlb200_qm_generate ----
    static void read_dct_params(BitReader &br, float (&out)[3][17], int &n) {
        n = 1 + (int)br.bits(4);
        for (int c = 0; c < 3; c++) {
            for (int i = 0; i < n; i++) out[c][i] = br.f16();
            out[c][0] *= 64.0f;
        }
    }
    void read_hf_global(FrameData &f, BitReader &br) {
        f.quant_all_default = br.flag();
        if (!f.quant_all_default) {
            for (int i = 0; i < 17; i++) {
                QuantParams &q = f.qparams[i];
                q = QuantParams();
                q.mode = (int)br.bits(3);
                if (q.mode == 7) coverage().raw_quant++; else if (q.mode != 0) coverage().custom_quant++;
                const bool small = (i >= 0 && i <= 3) || i == 9 || i == 10;
                if (!(q.mode == 0 || q.mode == 6 || q.mode == 7) && !small) throw StreamError("quant table encoding does not fit its transform");
                switch (q.mode) {
                case 0: break;                                         // library default
                case 1:                                                // Hornuss
                    q.n_param = 3;
                    for (int c = 0; c < 3; c++) for (int k = 0; k < 3; k++) q.param[c][k] = 64.0f * br.f16();
                    break;
                case 2:                                                // DCT2
                    q.n_param = 6;
                    for (int c = 0; c < 3; c++) for (int k = 0; k < 6; k++) q.param[c][k] = 64.0f * br.f16();
                    break;
                case 3:                                                // DCT4
                    q.n_param = 2;
                    for (int c = 0; c < 3; c++) for (int k = 0; k < 2; k++) q.param[c][k] = 64.0f * br.f16();
                    read_dct_params(br, q.dct_param, q.n_dct);
                    break;
                case 4:                                                // DCT4x8
                    q.n_param = 1;
                    for (int c = 0; c < 3; c++) q.param[c][0] = br.f16();
                    read_dct_params(br, q.dct_param, q.n_dct);
                    break;
                case 5:                                                // AFV
                    q.n_param = 9;
                    for (int c = 0; c < 3; c++)
                        for (int k = 0; k < 9; k++) {
                            q.param[c][k] = br.f16();
                            if (k < 6) q.param[c][k] *= 64.0f;
                        }
                    read_dct_params(br, q.dct_param, q.n_dct);
                    read_dct_params(br, q.params4x4, q.n_4x4);
                    break;
                case 6: read_dct_params(br, q.dct_param, q.n_dct); break;
                default: {                                             // raw: three matrixH x matrixW channels, modular coded
                    q.denominator = br.f16();
                    const int mh = kParamShape[i][0], mw = kParamShape[i][1];
                    std::vector<Channel> info;
                    for (int c = 0; c < 3; c++) info.emplace_back(mh, mw, 0, 0);
                    ModularStream ms;
                    ms.init(br, fc_, 1 + 3 * f.num_lf_groups + i, std::move(info));
                    ms.decode_channels(br);
                    if (ms.channels.size() != 3) throw StreamError("raw quant table stream must end with three channels");
                    for (int c = 0; c < 3; c++) {
                        q.raw[c].resize((size_t)mh * mw);
                        for (size_t k = 0; k < q.raw[c].size(); k++) q.raw[c][k] = (float)ms.channels[c].px[k];
                    }
                }
                }
            }
        }
        num_hf_presets_ = 1 + (int)br.bits(ceil_log1p((uint64_t)f.num_groups - 1));
    }

    // ---- passes (Pass.java, HFPass.java) ----
    static const std::vector<uint32_t> &natural_order(int order_id) {
        // all 13 tables are built once, under the function-static's initialisation lock: two threads parsing at once
        // (ctypes releases the GIL) can never see a half-filled table
        static const std::array<std::vector<uint32_t>, 13> cache = [] {
            std::array<std::vector<uint32_t>, 13> t;
            for (int b = 0; b < 13; b++) t[b] = build_natural_order(b);
            return t;
        }();
        return cache[order_id];
    }
    static std::vector<uint32_t> build_natural_order(int order_id) {
        std::vector<uint32_t> o;
        const int H = kOrderShape[order_id][0], W = kOrderShape[order_id][1], bh = H >> 3, bw = W >> 3, md = std::max(bh, bw);
        struct Key { int llf, k1, k2; uint32_t pos; };
        std::vector<Key> keys;
        keys.reserve((size_t)H * W);
        for (int y = 0; y < H; y++)
            for (int x = 0; x < W; x++) {
                Key k;
                k.pos = ((uint32_t)y << 16) | (uint32_t)x;
                if (y < bh && x < bw) {
                    k.llf = 0; k.k1 = y; k.k2 = x;
                } else {
                    const int sy = y * md / bh, sx = x * md / bw;
                    k.llf = 1;
                    k.k1 = sy + sx;
                    k.k2 = (k.k1 & 1) ? sy - sx : sx - sy;
                }
                keys.push_back(k);
            }
        std::sort(keys.begin(), keys.end(), [](const Key &a, const Key &b) {
            if (a.llf != b.llf) return a.llf < b.llf;
            if (a.k1 != b.k1) return a.k1 < b.k1;
            return a.k2 < b.k2;
        });
        o.resize(keys.size());
        for (size_t i = 0; i < keys.size(); i++) o[i] = keys[i].pos;
        return o;
    }
    void read_passes(FrameData &f, BitReader &br) {
        const FrameHeader &h = f.hdr;
        passes_.assign(h.num_passes, PassState());
        for (int p = 0; p < h.num_passes; p++) {
            PassState &ps = passes_[p];
            ps.max_shift = p > 0 ? passes_[p - 1].min_shift : 3;
            int n = -1;
            if (h.passes_coded)
                for (int i = 0; i <= h.num_ds; i++)
                    if (h.last_pass[i] == p) { n = i; break; }
            ps.min_shift = n >= 0 ? ceil_log1p((uint64_t)h.downsample[n] - 1) : ps.max_shift;
            for (size_t i = 0; i < f.modular.channels.size(); i++) {
                const Channel &c = f.modular.channels[i];
                if (c.decoded) continue;
                const int m = std::min(c.vshift, c.hshift);
                if (ps.min_shift <= m && m < ps.max_shift) ps.replaced.push_back((int)i);
            }
            if (h.encoding != ENC_VARDCT) continue;
            const uint32_t used = br.u32(0x5f, 0, 0x13, 0, 0, 0, 0, 13);
            if (used) coverage().coded_orders++;
            EntropyStream es;
            if (used) es = EntropyStream(br, 8);
            for (int b = 0; b < 13; b++) {
                const std::vector<uint32_t> &nat = natural_order(b);
                for (int c = 0; c < 3; c++) {
                    if (used >> b & 1) {
                        const std::vector<uint32_t> perm = read_permutation(br, es, (uint32_t)nat.size(), (uint32_t)nat.size() / 64);
                        ps.order[b][c].resize(nat.size());
                        for (size_t i = 0; i < nat.size(); i++) ps.order[b][c][i] = nat[perm[i]];
                    } else {
                        ps.order[b][c].clear();       // natural
                    }
                }
            }
            if (used) es.expect_final_state("coefficient order permutations");
            ps.coeff_stream = EntropyStream(br, 495 * num_hf_presets_ * num_block_clusters_);
        }
    }

    // ---- pass groups (Frame.java:317-374, PassGroup.java:67-84) ----
    void decode_pass_groups(FrameData &f) {
        const FrameHeader &h = f.hdr;
        for (int b = 0; b < 13; b++) natural_order(b);       // fill the shared cache before any task reads it
        for (int p = 0; p < h.num_passes; p++) {               // passes add into the same coefficients: one after the other
            for (int idx : passes_[p].replaced) f.modular.channels[idx].allocate();
            parallel_sections(f.num_groups, [&](int g) {
                BitReader &br = section(2 + f.num_lf_groups + (size_t)p * f.num_groups + g);
                if (h.encoding == ENC_VARDCT) read_hf_coefficients(f, br, p, g);
                ModularStream ms;
                ms.init(br, fc_, 18 + 3 * f.num_lf_groups + f.num_groups * p + g, cut_channels(f, passes_[p].replaced, g, h.group_dim));
                ms.decode_channels(br);
                paste_channels(f, passes_[p].replaced, ms);
            });
        }
    }

    // HFCoefficients.java:49-138 (+ context helpers :230-265).  Passes are summed into f.qcoeff (PassGroup.java:174-200).
    void read_hf_coefficients(FrameData &f, BitReader &br, int pass, int group) {
        static const int8_t kFreqCtx[64] = {-1, 0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 15, 16, 16, 17, 17, 18, 18, 19, 19, 20, 20, 21, 21, 22, 22,
                                            23, 23, 23, 23, 24, 24, 24, 24, 25, 25, 25, 25, 26, 26, 26, 26, 27, 27, 27, 27, 28, 28, 28, 28, 29, 29, 29, 29, 30, 30, 30, 30};
        static const int16_t kNzCtx[64] = {-1, 0, 31, 62, 62, 93, 93, 93, 93, 123, 123, 123, 123, 152, 152, 152, 152, 152, 152, 152, 152, 180, 180, 180, 180, 180,
                                           180, 180, 180, 180, 180, 180, 180, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206,
                                           206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206, 206};
        static const int kOrderC[3] = {1, 0, 2};
        const FrameHeader &h = f.hdr;
        PassState &ps = passes_[pass];
        const int preset = (int)br.bits(ceil_log1p((uint64_t)num_hf_presets_ - 1));
        const int offset = 495 * num_block_clusters_ * preset;
        const int shift = h.pass_shift[pass];
        const int grow = group / f.group_cols, gcol = group % f.group_cols;
        const int lfg_id = (grow >> 3) * f.lf_group_cols + (gcol >> 3);
        const LFGroupState &st = lfg_[lfg_id];
        const int gpy = (grow & 7) << 5, gpx = (gcol & 7) << 5;       // group origin inside its LF group, in blocks
        int32_t nz[3][32][32];
        std::memset(nz, 0, sizeof nz);
        EntropyStream es = ps.coeff_stream.fork();
        for (uint32_t b : st.blocks) {
            const int by = (int)(b >> 16), bx = (int)(b & 0xffff);
            const int gy = by - gpy, gx = bx - gpx;
            if (gy < 0 || gx < 0 || gy >= 32 || gx >= 32) continue;
            const int type = st.dct_select[(size_t)by * st.bw + bx];
            const TType &tt = kTypes[type];
            const bool flip = type_flips(type);
            const int32_t hf_mul = st.hf_mul[(size_t)by * st.bw + bx];
            const int lf_index = st.lf_index[(size_t)by * st.bw + bx];
            const int bh = tt.ph >> 3, bw = tt.pw >> 3, num_blocks = bh * bw;
            for (int c : kOrderC) {
                const int sgy = gy >> h.shift_y[c], sgx = gx >> h.shift_x[c];
                if (gy != sgy << h.shift_y[c] || gx != sgx << h.shift_x[c]) continue;
                // predicted non-zero count (:258-265)
                int predicted;
                if (sgx == 0 && sgy == 0) predicted = 32;
                else if (sgx == 0) predicted = nz[c][sgy - 1][0];
                else if (sgy == 0) predicted = nz[c][0][sgx - 1];
                else predicted = (nz[c][sgy - 1][sgx] + nz[c][sgy][sgx - 1] + 1) >> 1;
                // block context (:230-239)
                int idx = (c < 2 ? 1 - c : c) * 13 + tt.order_id;
                idx *= (int)qf_thresholds_.size() + 1;
                for (int32_t t : qf_thresholds_) idx += hf_mul > t;
                idx *= num_lf_contexts_;
                const int block_ctx = block_ctx_map_.at((size_t)idx + lf_index);
                const int pred_c = std::min(predicted, 64);
                const int nz_ctx = offset + block_ctx + num_block_clusters_ * (pred_c < 8 ? pred_c : 4 + pred_c / 2);
                int32_t non_zero = (int32_t)es.read(br, nz_ctx);
                const int32_t per_block = (non_zero + num_blocks - 1) / num_blocks;
                for (int iy = 0; iy < bh; iy++)
                    for (int ix = 0; ix < bw; ix++) {
                        if (sgy + iy < 32 && sgx + ix < 32) nz[c][sgy + iy][sgx + ix] = per_block;
                    }
                if (non_zero <= 0) continue;
                const std::vector<uint32_t> &order = ps.order[tt.order_id][c].empty() ? natural_order(tt.order_id) : ps.order[tt.order_id][c];
                const int order_size = (int)order.size();
                const int hist_ctx = offset + 458 * block_ctx + 37 * num_block_clusters_;
                // frame-level destination of this group's coefficient rectangle for channel c
                const int cw = f.padded_w >> h.shift_x[c];
                const int py0 = ((grow << 8) >> h.shift_y[c]) + (sgy << 3), px0 = ((gcol << 8) >> h.shift_x[c]) + (sgx << 3);
                if (py0 + tt.ph > (f.padded_h >> h.shift_y[c]) || px0 + tt.pw > cw) throw StreamError("varblock leaves its (subsampled) plane");
                int32_t *plane = f.qcoeff[c].data();
                uint32_t prev_sym = 0;
                for (int k = 0; k < order_size - num_blocks; k++) {
                    const int prev = k == 0 ? (non_zero > order_size / 16 ? 0 : 1) : (prev_sym != 0 ? 1 : 0);
                    const int nzb = (non_zero + num_blocks - 1) / num_blocks;
                    if (nzb > 63) throw StreamError("non-zero count out of range");
                    const int ctx = hist_ctx + (kNzCtx[nzb] + kFreqCtx[(k + num_blocks) / num_blocks]) * 2 + prev;
                    const uint32_t u = es.read(br, ctx);
                    prev_sym = u;
                    const uint32_t o = order[k + num_blocks];
                    const int oy = (int)(o >> 16), ox = (int)(o & 0xffff);
                    const int py = py0 + (flip ? ox : oy), px = px0 + (flip ? oy : ox);
                    int32_t &dst = plane[(size_t)py * cw + px];
                    dst = detail::wrap_add(dst, detail::wrap_shl(unpack_signed(u), shift));
                    if (u != 0 && --non_zero == 0) break;
                }
                if (non_zero != 0) throw StreamError("coefficients ran out before the non-zero count did");
            }
        }
        es.expect_final_state("HF coefficients");
    }
};

}  // namespace jxlf
