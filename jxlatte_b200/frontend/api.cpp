// api.cpp -- C ABI of the host front end (libjxlfront.so): .jxl bytes -> headers (as one JSON document) + the
// post-entropy arrays of every frame, addressed by name.  Declared in include/jxlfront.h.
//
// This is the sequential half of jxlatte's decoder (JXLCodestreamDecoder.decode's header/frame loop,
// J/JXLCodestreamDecoder.java:539-626) restated in C++; the data-parallel half is libjxlb200.so.
#include <cstdio>
#include <sstream>

#include <omp.h>

#include "frame.hpp"
#include "../../include/jxlfront.h"

using namespace jxlf;

struct jxlf_image {
    std::vector<uint8_t> codestream;
    ImageHeader ih;
    std::vector<std::unique_ptr<FrameData>> frames;
    std::string json, error;
    int status = 0;
    bool lf_only = false;
};

namespace {

struct Json {
    std::ostringstream o;
    bool first = true;
    void sep() { if (!first) o << ","; first = false; }
    void key(const char *k) { sep(); o << "\"" << k << "\":"; }
    template <class T> void num(const char *k, T v) { key(k); o << v; }
    void flt(const char *k, float v) { key(k); char b[40]; std::snprintf(b, sizeof b, "%.9g", (double)v); o << b; }
    void boolean(const char *k, bool v) { key(k); o << (v ? "true" : "false"); }
    void str(const char *k, const std::string &v) {
        key(k);
        o << "\"";
        for (unsigned char c : v) {
            if (c == '"' || c == '\\') o << '\\' << c;
            else if (c < 0x20 || c >= 0x7f) { char b[8]; std::snprintf(b, sizeof b, "\\u%04x", c); o << b; }
            else o << c;
        }
        o << "\"";
    }
    template <class It> void farr(const char *k, It b, It e) {
        key(k); o << "[";
        for (It i = b; i != e; ++i) { if (i != b) o << ","; char t[40]; std::snprintf(t, sizeof t, "%.9g", (double)*i); o << t; }
        o << "]";
    }
    template <class It> void iarr(const char *k, It b, It e) {
        key(k); o << "[";
        for (It i = b; i != e; ++i) { if (i != b) o << ","; o << (long long)*i; }
        o << "]";
    }
    void open(const char *k, char br) { if (k) key(k); else sep(); o << br; first = true; }
    void close(char br) { o << br; first = false; }
};

void describe(jxlf_image &im) {
    Json j;
    const ImageHeader &ih = im.ih;
    j.open(nullptr, '{');
    j.num("width", ih.width); j.num("height", ih.height); j.num("level", ih.level); j.num("orientation", ih.orientation);
    j.num("bits_per_sample", ih.depth.bits); j.num("exp_bits", ih.depth.exp_bits); j.boolean("float_samples", ih.depth.is_float);
    j.boolean("xyb_encoded", ih.xyb_encoded); j.boolean("modular_16bit", ih.modular_16bit);
    j.num("color_channels", ih.color_channels());
    j.boolean("have_animation", ih.have_animation);
    j.open("color", '{');
    j.boolean("use_icc", ih.color.use_icc); j.num("color_space", ih.color.color_space); j.num("white_point", ih.color.white_point);
    j.num("primaries", ih.color.primaries); j.num("transfer", ih.color.transfer); j.num("rendering_intent", ih.color.rendering_intent);
    j.farr("white_xy", ih.color.white_xy, ih.color.white_xy + 2);
    j.farr("prim_xy", &ih.color.prim_xy[0][0], &ih.color.prim_xy[0][0] + 6);
    j.close('}');
    j.flt("intensity_target", ih.intensity_target); j.flt("min_nits", ih.min_nits);
    j.farr("opsin_inverse", ih.opsin_inv, ih.opsin_inv + 9); j.farr("opsin_bias", ih.opsin_bias, ih.opsin_bias + 3);
    j.farr("quant_bias", ih.quant_bias, ih.quant_bias + 3); j.flt("quant_bias_numerator", ih.quant_bias_numerator);
    j.farr("up2", ih.up2.begin(), ih.up2.end()); j.farr("up4", ih.up4.begin(), ih.up4.end()); j.farr("up8", ih.up8.begin(), ih.up8.end());
    j.num("icc_bytes", ih.encoded_icc.size());
    j.open("extra_channels", '[');
    for (auto &e : ih.extra) {
        j.open(nullptr, '{');
        j.num("type", e.type); j.num("bits_per_sample", e.depth.bits); j.num("exp_bits", e.depth.exp_bits); j.num("dim_shift", e.dim_shift);
        j.str("name", e.name); j.boolean("alpha_associated", e.alpha_associated);
        j.close('}');
    }
    j.close(']');
    {
        Coverage &c = coverage();
        j.open("coverage", '{');
        j.num("entropy_streams", c.streams.load()); j.num("ans", c.ans_streams.load()); j.num("prefix", c.prefix_streams.load());
        j.num("lz77_streams", c.lz77_streams.load()); j.num("lz77_copies", c.lz77_copies.load()); j.num("mtf_context_maps", c.mtf_context_maps.load());
        j.num("permuted_toc", c.permuted_toc.load()); j.num("coded_coefficient_orders", c.coded_orders.load());
        j.num("multi_pass_frames", c.multi_pass_frames.load()); j.num("custom_block_contexts", c.custom_block_ctx.load());
        j.num("weighted_predictor_channels", c.wp_channels.load()); j.num("global_trees", c.global_trees.load()); j.num("local_trees", c.local_trees.load());
        j.num("squeeze", c.squeeze.load()); j.num("palette", c.palette.load()); j.num("delta_palette", c.delta_palette.load()); j.num("rct", c.rct.load());
        j.num("raw_quant_tables", c.raw_quant.load()); j.num("custom_quant_tables", c.custom_quant.load()); j.num("lf_smoothing_groups", c.lf_smoothing.load());
        j.close('}');
    }
    j.open("frames", '[');
    for (auto &fp : im.frames) {
        const FrameData &f = *fp;
        const FrameHeader &h = f.hdr;
        j.open(nullptr, '{');
        j.num("type", h.type); j.num("encoding", h.encoding); j.num("flags", (unsigned long long)h.flags); j.boolean("do_ycbcr", h.do_ycbcr);
        j.iarr("shift_x", h.shift_x, h.shift_x + 3); j.iarr("shift_y", h.shift_y, h.shift_y + 3);
        j.num("upsampling", h.upsampling); j.iarr("ec_upsampling", h.ec_upsampling.begin(), h.ec_upsampling.end());
        j.num("group_dim", h.group_dim); j.num("xqm_scale", h.xqm_scale); j.num("bqm_scale", h.bqm_scale);
        j.num("num_passes", h.num_passes); j.num("lf_level", h.lf_level);
        j.num("x0", h.x0); j.num("y0", h.y0); j.num("width", h.width); j.num("height", h.height);
        j.num("padded_width", f.padded_w); j.num("padded_height", f.padded_h);
        j.num("blend_mode", h.blending.mode); j.num("blend_source", h.blending.source); j.num("blend_alpha", h.blending.alpha_channel);
        j.boolean("blend_clamp", h.blending.clamp);
        j.num("duration", h.duration); j.boolean("is_last", h.is_last); j.num("save_as_reference", h.save_as_reference);
        j.boolean("save_before_ct", h.save_before_ct); j.str("name", h.name);
        j.boolean("gab", h.rf.gab); j.farr("gab_w1", h.rf.gab_w1, h.rf.gab_w1 + 3); j.farr("gab_w2", h.rf.gab_w2, h.rf.gab_w2 + 3);
        j.num("epf_iters", h.rf.epf_iters); j.farr("epf_sharp_lut", h.rf.sharp_lut, h.rf.sharp_lut + 8);
        j.farr("epf_channel_scale", h.rf.channel_scale, h.rf.channel_scale + 3);
        j.flt("epf_pass0_sigma_scale", h.rf.pass0_sigma_scale); j.flt("epf_pass2_sigma_scale", h.rf.pass2_sigma_scale);
        j.flt("epf_border_sad_mul", h.rf.border_sad_mul); j.flt("epf_sigma_for_modular", h.rf.sigma_for_modular);
        j.num("toc_bit_offset", (unsigned long long)f.toc_bit_offset); j.num("toc_first_section", (unsigned long long)f.toc_first_section);
        j.iarr("toc_lengths", f.toc_lengths.begin(), f.toc_lengths.end());
        j.num("num_groups", f.num_groups); j.num("num_lf_groups", f.num_lf_groups);
        j.farr("lf_dequant", f.lf_dequant, f.lf_dequant + 3); j.farr("scaled_dequant", f.scaled_dequant, f.scaled_dequant + 3); j.num("global_scale", f.global_scale); j.num("quant_lf", f.quant_lf);
        j.num("color_factor", f.color_factor); j.flt("base_corr_x", f.base_corr_x); j.flt("base_corr_b", f.base_corr_b);
        j.num("x_factor_lf", f.x_factor_lf); j.num("b_factor_lf", f.b_factor_lf);
        j.farr("noise", f.noise, f.noise + 8); j.num("num_patches", f.num_patches); j.num("num_splines", f.num_splines);
        j.open("patches", '[');
        for (auto &pt : f.patches) {
            j.open(nullptr, '{');
            j.num("ref", pt.ref); j.num("x0", pt.x0); j.num("y0", pt.y0); j.num("w", pt.w); j.num("h", pt.h);
            j.iarr("pos", pt.pos.begin(), pt.pos.end()); j.iarr("blend", pt.blend.begin(), pt.blend.end());
            j.close('}');
        }
        j.close(']');
        j.num("spline_quant_adjust", f.spline_quant_adjust);
        j.open("splines", '[');
        for (auto &sp : f.splines) {
            j.open(nullptr, '{');
            j.iarr("points", sp.points.begin(), sp.points.end());
            j.iarr("coeff", &sp.coeff[0][0], &sp.coeff[0][0] + 128);
            j.close('}');
        }
        j.close(']');
        j.open("ec_blending", '[');
        for (auto &b : h.ec_blending) {
            j.open(nullptr, '[');
            j.sep(); j.o << b.mode;
            j.sep(); j.o << b.alpha_channel;
            j.sep(); j.o << (b.clamp ? 1 : 0);
            j.sep(); j.o << b.source;
            j.close(']');
        }
        j.close(']');
        j.boolean("decoded", !f.dct_select.empty() || !f.lf[0].empty() || f.has_modular || h.encoding == ENC_MODULAR);
        if (!f.lf_only) j.boolean("quant_all_default", f.quant_all_default);      // HfGlobal: not read by an LF-only parse
        if (!f.lf_only && !f.quant_all_default) {
            j.open("quant_params", '[');
            for (const QuantParams &q : f.qparams) {
                j.open(nullptr, '{');
                j.num("mode", q.mode); j.num("n_dct", q.n_dct); j.num("n_param", q.n_param); j.num("n_4x4", q.n_4x4); j.flt("denominator", q.denominator);
                j.farr("dct_param", &q.dct_param[0][0], &q.dct_param[0][0] + 51); j.farr("param", &q.param[0][0], &q.param[0][0] + 27);
                j.farr("params4x4", &q.params4x4[0][0], &q.params4x4[0][0] + 51);
                j.close('}');
            }
            j.close(']');
        }
        j.open("modular", '{');
        j.num("nb_meta", f.modular.nb_meta); j.boolean("transformed", f.modular.transformed);
        j.open("channels", '[');
        for (auto &c : f.modular.channels) {
            j.open(nullptr, '{');
            j.num("h", c.h); j.num("w", c.w); j.num("hshift", c.hshift); j.num("vshift", c.vshift);
            j.close('}');
        }
        j.close(']');
        j.open("transforms", '[');
        for (auto &t : f.modular.transforms) {
            j.open(nullptr, '{');
            j.num("tr", t.tr); j.num("begin_c", t.begin_c); j.num("rct_type", t.rct_type); j.num("num_c", t.num_c);
            j.num("nb_colors", t.nb_colors); j.num("nb_deltas", t.nb_deltas); j.num("d_pred", t.d_pred);
            j.open("sp", '[');
            for (auto &s : t.sp) {
                j.open(nullptr, '[');
                j.sep(); j.o << (s.horizontal ? 1 : 0);
                j.sep(); j.o << (s.in_place ? 1 : 0);
                j.sep(); j.o << s.begin_c;
                j.sep(); j.o << s.num_c;
                j.close(']');
            }
            j.close(']');
            j.close('}');
        }
        j.close(']');
        j.close('}');
        j.close('}');
    }
    j.close(']');
    if (im.lf_only) j.boolean("lf_only", true);
    j.close('}');
    im.json = j.o.str();
}

}  // namespace

extern "C" {

// flags: bit 0 = also undo the frame-level modular transforms on the host (tests / cross-checks; the product path
// leaves them to the GPU), bit 1 = stop after the headers of the first frame, bit 2 = parse every frame up to its LF groups only.
int32_t jxlf_decode(const uint8_t *data, uint64_t size, int32_t flags, jxlf_image **out) {
    if (!data || !out) return -1;
    auto im = std::make_unique<jxlf_image>();
    coverage().reset();
    im->lf_only = (flags & JXLF_LF_ONLY) != 0;
    try {
        // the host transforms need every channel, and an LF-only parse leaves the pass groups' channels empty
        if ((flags & JXLF_HOST_TRANSFORMS) && im->lf_only) throw std::invalid_argument("JXLF_HOST_TRANSFORMS with JXLF_LF_ONLY");
        std::vector<uint8_t> file(data, data + size);
        const int level = extract_codestream(file, im->codestream);
        BitReader br(im->codestream.data(), im->codestream.size());
        im->ih.read(br, level);
        if (im->ih.preview_h) throw Unsupported("preview frames");
        while (true) {
            auto f = std::make_unique<FrameData>();
            FrameDecoder dec(br, im->ih);
            dec.read_header(*f);
            if (flags & 2) { im->frames.push_back(std::move(f)); break; }
            dec.decode(*f, im->lf_only);
            if (flags & 1) f->modular.apply_transforms();
            const bool last = f->hdr.is_last;
            im->frames.push_back(std::move(f));
            if (last) break;
        }
    } catch (const Unsupported &e) {
        im->status = -3;
        im->error = e.what();
    } catch (const StreamError &e) {
        im->status = -2;
        im->error = e.what();
    } catch (const std::exception &e) {
        im->status = -1;
        im->error = e.what();
    }
    describe(*im);
    const int32_t st = im->status;
    *out = im.release();
    return st;
}

void jxlf_free(jxlf_image *im) { delete im; }
void jxlf_set_threads(int32_t n) { if (n >= 1) omp_set_num_threads(n); }
const char *jxlf_error(const jxlf_image *im) { return im ? im->error.c_str() : "null image"; }
const char *jxlf_describe(const jxlf_image *im) { return im ? im->json.c_str() : "{}"; }

// Arrays by name.  dtype: 0 int32, 1 float32, 2 uint8.  Returns 0, or -1 when there is no such array.
//   qcoeff/lf (index = channel), dct_select, block_origin, hf_mul, sharpness, x_from_y, b_from_y,
//   modular (index = channel of the frame-level modular stream), qraw (index = 3 * parameter set + channel), icc
int32_t jxlf_array(const jxlf_image *im, int32_t frame, const char *name, int32_t index, const void **ptr, int64_t *count, int32_t *dtype) {
    if (!im || !name || !ptr || !count || !dtype) return -1;
    const std::string n(name);
    if (n == "icc") { *ptr = im->ih.encoded_icc.data(); *count = (int64_t)im->ih.encoded_icc.size(); *dtype = 2; return 0; }
    if (frame < 0 || frame >= (int)im->frames.size()) return -1;
    const FrameData &f = *im->frames[frame];
    auto give = [&](const auto &v, int dt) { *ptr = v.data(); *count = (int64_t)v.size(); *dtype = dt; return 0; };
    if (f.lf_only && (n == "qcoeff" || n == "dct_select" || n == "block_origin" || n == "hf_mul" || n == "sharpness" || n == "x_from_y" ||
                      n == "b_from_y"))
        return -1;                                       // HF state: an LF-only parse never read it
    if (n == "qcoeff" && index >= 0 && index < 3) return give(f.qcoeff[index], 0);
    if (n == "lf" && index >= 0 && index < 3) return give(f.lf[index], 1);
    if (n == "lf_quant" && index >= 0 && index < 3) return give(f.lf_quant[index], 0);
    if (n == "lf_extra_precision") return give(f.lf_extra_precision, 2);
    if (n == "dct_select") return give(f.dct_select, 2);
    if (n == "block_origin") return give(f.block_origin, 2);
    if (n == "hf_mul") return give(f.hf_mul, 0);
    if (n == "sharpness") return give(f.sharpness, 0);
    if (n == "x_from_y") return give(f.x_from_y, 0);
    if (n == "b_from_y") return give(f.b_from_y, 0);
    if (n == "modular" && index >= 0 && index < (int)f.modular.channels.size()) return give(f.modular.channels[index].px, 0);
    if (n == "qraw" && index >= 0 && index < 51) return give(f.qparams[index / 3].raw[index % 3], 1);
    return -1;
}

}  // extern "C"
