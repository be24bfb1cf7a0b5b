// The model graph of the hot path, appended op by op to a Plan (static shapes => one CUDA graph).
//
// Mirrors, layer for layer, what the reference executes through diffusers 0.25.1:
//   VAE encoder  : my_vae_encoder_fwd        /root/reference/src/model.py:14-27   (+ quant_conv, posterior sample)
//   UNet         : UNet2DConditionModel call /root/reference/src/pix2pix_turbo.py:199 (SD-Turbo config, t == 999)
//   DDPM step    : sched.step                /root/reference/src/pix2pix_turbo.py:200 (closed form)
//   VAE decoder  : my_vae_decoder_fwd        /root/reference/src/model.py:30-54   (skip convs, gamma)
// with LoRA folded into the weights, the time embedding folded into conv1 biases, TwinConv blended, and
// NHWC activations so that [B,H,W,C] == [B, HW, C] tokens (no permutes around the transformer blocks).
#include "engine.cuh"

namespace i2it {

static inline int ceil_div_i(long long a, long long b) { return static_cast<int>((a + b - 1) / b); }

#define DISPATCH_T(dt, ...)                                   \
  do {                                                        \
    if ((dt) == DT_BF16) { using T = __nv_bfloat16; __VA_ARGS__; } \
    else { using T = __half; __VA_ARGS__; }                   \
  } while (0)

// ------------------------------------------------------------------------------------------ VAE
Act Engine::vae_resnet(Plan& P, const std::string& p, const Act& x, const Act* skip, const PW* skip_w, bool gn_next) {
  Act h = group_norm(P, x, norm(p + ".norm1"), 1e-6f, true);
  ConvOpts o1; o1.gn_out = true;                     // conv1 feeds norm2: its epilogue takes the GroupNorm statistics
  h = conv(P, h, prep(p + ".conv1", {p + ".conv1"}), o1);
  h = group_norm(P, h, norm(p + ".norm2"), 1e-6f, true);
  ConvOpts o;
  o.gn_out = gn_next;                                // the block's output feeds another GroupNorm (norm1 / attention / conv_norm_out)
  if (has(p + ".conv_shortcut.weight")) {
    // x + conv2(h) with a 1x1 shortcut: the shortcut is one more K-slab of the SAME GEMM (second A tensor), its bias is
    // pre-added to conv2's, so there is no separate launch and no residual read
    I2IT_CHECK(skip == nullptr, "vae_resnet: shortcut and skip source at once");
    PW wsc = prep(p + ".conv_shortcut", {p + ".conv_shortcut"});
    PW w2 = prep(p + ".conv2+sc", {p + ".conv2"}, false, 1.f, raw(p + ".conv_shortcut", "bias").d);
    o.x2 = &x; o.w2 = &wsc;
    return conv(P, h, w2, o);
  }
  o.res = &x;
  if (skip) { o.x2 = skip; o.w2 = skip_w; }        // decoder: the next block's  + skip_conv(skip*gamma)  folded in here
  return conv(P, h, prep(p + ".conv2", {p + ".conv2"}), o);
}

Act Engine::vae_attn(Plan& P, const std::string& p, const Act& x) {
  // diffusers Attention (1 head, d = C) with residual; tokens are the NHWC pixels
  const int C = x.C, B = x.N, N = x.H * x.W;
  Act t = group_norm(P, x, norm(p + ".group_norm"), 1e-6f, false);
  Act qk = linear(P, t, prep(p + ".qk", {p + ".to_q", p + ".to_k"}));
  Act vt = vt_proj(P, t, B, N, prep(p + ".to_v", {p + ".to_v"}));
  Act a = attention(P, qk.slice(0, C), qk.slice(C, C), vt, B, N, N, 1, C, B);
  a.N = x.N; a.H = x.H; a.W = x.W;
  return linear(P, a, prep(p + ".to_out.0", {p + ".to_out.0"}), &x, TG_ACT_NONE, true);   // -> mid_block.resnets.1.norm1
}

Act Engine::build_vae_encoder(Plan& P, const std::string& vp, int B, int H, int W, std::vector<Act>& skips, bool u8_in) {
  const std::string e = vp + "encoder";
  // conv_in (3 -> C0, 3x3): the NCHW boundary tensor is packed straight into im2col rows [B,H,W,32] (27 taps*channels + 5
  // zeros), so the conv is ONE K=32 GEMM tap with 64-byte TMA rows instead of nine taps of 16-byte rows
  Act xcol = alloc_act(P, B, H, W, 32);
  {
    const long long total = static_cast<long long>(H) * W * B;
    uint16_t* yp = xcol.p;
    Plan* plan = &P;
    const int dt = dtype, hh = H, ww = W;
    if (u8_in) {
      add_op(P, [=](cudaStream_t st) {
        DISPATCH_T(dt, (launch_k(pack_input_im2col_u8_kernel<T>, dim3(ceil_div_i(total, 128)), dim3(128), 0, st, 0,
                           reinterpret_cast<const uint8_t*>(plan->io.x_u8), reinterpret_cast<T*>(yp), hh, ww, total, plan->io.in_mode)));
      }, "pack_im2col_u8", 0, 1.0 * total * (3 + 64));
    } else {
      add_op(P, [=](cudaStream_t st) {
        DISPATCH_T(dt, (launch_k(pack_input_im2col_kernel<T>, dim3(ceil_div_i(total, 128)), dim3(128), 0, st, 0,
                           reinterpret_cast<const T*>(plan->io.x), reinterpret_cast<T*>(yp), hh, ww, total)));
      }, "pack_im2col", 0, 2.0 * total * (3 + 32));
    }
  }
  ConvOpts oin; oin.ksize = 1; oin.gn_out = true;
  Act s = conv(P, xcol, prep_im2col3(e + ".conv_in"), oin);
  xcol = Act();
  for (int i = 0; i < 4; ++i) {
    skips.push_back(s);                                   // model.py:18-20: the INPUT of each down block
    mark(P, "skip" + std::to_string(i), s);
    for (int j = 0; j < 2; ++j)      // the last resnet before a downsampler feeds a conv, not a GroupNorm
      s = vae_resnet(P, e + ".down_blocks." + std::to_string(i) + ".resnets." + std::to_string(j), s, nullptr, nullptr,
                     !(j == 1 && i < 3));
    if (i < 3) {
      ConvOpts o; o.stride = 2; o.asym = true; o.gn_out = true;
      const std::string d = e + ".down_blocks." + std::to_string(i) + ".downsamplers.0.conv";
      s = conv(P, s, prep(d, {d}), o);
    }
  }
  s = vae_resnet(P, e + ".mid_block.resnets.0", s);
  s = vae_attn(P, e + ".mid_block.attentions.0", s);
  s = vae_resnet(P, e + ".mid_block.resnets.1", s);
  mark(P, "enc_mid", s);
  s = group_norm(P, s, norm(e + ".conv_norm_out"), 1e-6f, true);
  s = conv(P, s, prep(e + ".conv_out", {e + ".conv_out"}), ConvOpts());
  ConvOpts o1; o1.ksize = 1;
  Act mom = conv(P, s, prep(vp + "quant_conv", {vp + "quant_conv"}), o1);
  mark(P, "moments", mom);
  Act z = alloc_act(P, B, H / 8, W / 8, 8, 8, true);
  {
    const long long HW = static_cast<long long>(H / 8) * (W / 8), total = HW * B;
    const uint16_t* mp = mom.p;
    const int ldm = mom.ld, dt = dtype;
    uint16_t* zp = z.p;
    Plan* plan = &P;
    const float sf = cfg.scaling_factor;
    P.keep.push_back(mom.hold);
    add_op(P, [=](cudaStream_t st) {
      DISPATCH_T(dt, (launch_k(latent_sample_kernel<T>, dim3(ceil_div_i(total, 128)), dim3(128), 0, st, 0,
                         reinterpret_cast<const T*>(mp), ldm, reinterpret_cast<const T*>(plan->io.eps),
                         reinterpret_cast<const T*>(plan->io.noise), plan->io.r, sf, reinterpret_cast<T*>(zp), HW, total)));
    });
  }
  mark(P, "latent", z);
  return z;
}

void Engine::build_vae_decoder(Plan& P, const std::string& vp, const Act& dec_in, std::vector<Act>& skips) {
  const std::string d = vp + "decoder";
  ConvOpts o1; o1.ksize = 1;
  Act s = conv(P, dec_in, prep(vp + "post_quant_conv", {vp + "post_quant_conv"}), o1);
  { ConvOpts oc; oc.gn_out = true; s = conv(P, s, prep(d + ".conv_in", {d + ".conv_in"}), oc); }
  // `sample = sample + skip_conv_i(skip_i * gamma)` (src/model.py:40-42) is folded into whichever conv PRODUCES `sample`
  // for up-block i: mid_block.resnets.1.conv2 for i = 0, the previous block's upsampler conv for i >= 1.  gamma is folded
  // into the bias-free 1x1 weights.
  auto skip_w = [&](int i) { const std::string sk = d + ".skip_conv_" + std::to_string(i + 1); return prep(sk, {sk}, false, skip_gamma_); };
  s = vae_resnet(P, d + ".mid_block.resnets.0", s);
  s = vae_attn(P, d + ".mid_block.attentions.0", s);
  {
    PW w0 = skip_w(0);
    s = vae_resnet(P, d + ".mid_block.resnets.1", s, &skips[3], &w0);
    skips[3] = Act();
  }
  mark(P, "dec_mid", s);
  for (int i = 0; i < 4; ++i) {
    for (int j = 0; j < 3; ++j)      // resnets.2 feeds the upsampler conv (i < 3) or conv_norm_out (i == 3)
      s = vae_resnet(P, d + ".up_blocks." + std::to_string(i) + ".resnets." + std::to_string(j), s, nullptr, nullptr,
                     !(j == 2 && i < 3));
    if (i < 3) {
      // Upsample2D: nearest-2x + conv3x3, as four parity-phase 2x2 convs on the low-res tensor (2.25x fewer FLOPs, the
      // upsampled tensor never exists); the next block's skip conv rides along as a second source at output resolution
      const std::string u = d + ".up_blocks." + std::to_string(i) + ".upsamplers.0.conv";
      PW wn = skip_w(i + 1);
      s = conv_up2x(P, s, prep_subpixel(u), &skips[2 - i], &wn, true);
      skips[2 - i] = Act();
    }
    mark(P, "dec_up" + std::to_string(i), s);
  }
  s = group_norm(P, s, norm(d + ".conv_norm_out"), 1e-6f, true);
  if (cfg.keep_stages) {   // tests compare the PRE-clamp image (BASELINE.md section 5): one extra launch, test mode only
    Act pre = conv(P, s, prep(d + ".conv_out", {d + ".conv_out"}), ConvOpts());
    mark(P, "pre_clamp", pre);
  }
  ConvOpts oo; oo.act = TG_ACT_CLAMP1; oo.to_io_out_nchw = true;
  conv(P, s, prep(d + ".conv_out", {d + ".conv_out"}), oo);
}

// ------------------------------------------------------------------------------------------ UNet
Act Engine::unet_resnet(Plan& P, const std::string& p, const Act& x, bool gn_next, const Act* out) {
  Act h = group_norm(P, x, norm(p + ".norm1"), 1e-5f, true);
  // t == 999 always: time_emb_proj(silu(emb)) is a per-channel constant -> part of conv1's bias
  ConvOpts o1; o1.gn_out = true;
  h = conv(P, h, prep(p + ".conv1", {p + ".conv1"}, false, 1.f, temb_bias(p)), o1);
  h = group_norm(P, h, norm(p + ".norm2"), 1e-5f, true);
  ConvOpts o;
  o.gn_out = gn_next;
  o.out = out;
  if (has(p + ".conv_shortcut.weight")) {
    PW wsc = prep(p + ".conv_shortcut", {p + ".conv_shortcut"});
    PW w2 = prep(p + ".conv2+sc", {p + ".conv2"}, false, 1.f, raw(p + ".conv_shortcut", "bias").d);
    o.x2 = &x; o.w2 = &wsc;
    return conv(P, h, w2, o);
  }
  o.res = &x;
  return conv(P, h, prep(p + ".conv2", {p + ".conv2"}), o);
}

Act Engine::unet_xformer(Plan& P, const std::string& p, const Act& x, int heads, int text_batch, bool gn_next, const Act* out) {
  const int C = x.C, B = x.N, N = x.H * x.W, d = C / heads;
  const std::string b = p + ".transformer_blocks.0";
  Act t = group_norm(P, x, norm(p + ".norm"), 1e-6f, false);
  t = linear(P, t, prep(p + ".proj_in", {p + ".proj_in"}));
  {  // self-attention
    Act n = layer_norm(P, t, norm(b + ".norm1"));
    Act qk = linear(P, n, prep(b + ".attn1.qk", {b + ".attn1.to_q", b + ".attn1.to_k"}));
    Act vt = vt_proj(P, n, B, N, prep(b + ".attn1.to_v", {b + ".attn1.to_v"}));
    Act a = attention(P, qk.slice(0, C), qk.slice(C, C), vt, B, N, N, heads, d, B);
    a.N = x.N; a.H = x.H; a.W = x.W;
    t = linear(P, a, prep(b + ".attn1.to_out.0", {b + ".attn1.to_out.0"}), &t);
  }
  {  // cross-attention over the 77 text tokens
    Act n = layer_norm(P, t, norm(b + ".norm2"));
    Act q = linear(P, n, prep(b + ".attn2.to_q", {b + ".attn2.to_q"}));
    Act k2, v2t;
    if (text_kv_) {                                   // computed once per prompt by i2it_set_text
      auto it = text_kv_->kv.find(b);
      I2IT_CHECK(it != text_kv_->kv.end(), "no cached text K/V for " + b);
      k2 = it->second.first; v2t = it->second.second;
    } else {
      k2 = linear(P, text_, prep(b + ".attn2.to_k", {b + ".attn2.to_k"}));
      v2t = vt_proj(P, text_, text_batch, 77, prep(b + ".attn2.to_v", {b + ".attn2.to_v"}));
    }
    Act a = attention(P, q, k2, v2t, B, N, 77, heads, d, text_batch);
    a.N = x.N; a.H = x.H; a.W = x.W;
    t = linear(P, a, prep(b + ".attn2.to_out.0", {b + ".attn2.to_out.0"}), &t);
  }
  {  // GEGLU feed-forward: h * gelu(g) fused into the first projection's epilogue (weight rows interleaved)
    Act n = layer_norm(P, t, norm(b + ".norm3"));
    Act g = linear(P, n, prep(b + ".ff.net.0.proj", {b + ".ff.net.0.proj"}, true), nullptr, TG_ACT_GEGLU);
    t = linear(P, g, prep(b + ".ff.net.2", {b + ".ff.net.2"}), &t);
  }
  return linear(P, t, prep(p + ".proj_out", {p + ".proj_out"}), &x, TG_ACT_NONE, gn_next, out);
}

// every transformer block of the UNet, in execution-independent fixed order (the cross-attention K/V^T cache is keyed by it)
std::vector<std::string> Engine::xformer_prefixes() const {
  std::vector<std::string> v;
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 2; ++j) v.push_back("unet.down_blocks." + std::to_string(i) + ".attentions." + std::to_string(j));
  v.push_back("unet.mid_block.attentions.0");
  for (int i = 1; i < 4; ++i)
    for (int j = 0; j < 3; ++j) v.push_back("unet.up_blocks." + std::to_string(i) + ".attentions." + std::to_string(j));
  return v;
}

// K = to_k(text), V^T = (to_v(text))^T of every cross-attention layer: 2 launches per block, run only when the prompt changes
void Engine::build_text_kv(TextKV& T) {
  Plan& P = T.plan;
  T.text = alloc_act(P, T.text_batch, 1, 77, cfg.cross_dim);
  {
    uint16_t* tp = T.text.p;
    const size_t bytes = static_cast<size_t>(T.text_batch) * 77 * cfg.cross_dim * 2;
    Plan* plan = &P;
    add_op(P, [=](cudaStream_t st) {
      cudaMemcpyAsync(tp, plan->io.text, bytes, cudaMemcpyDeviceToDevice, st);
    });
  }
  for (const auto& p : xformer_prefixes()) {
    const std::string b = p + ".transformer_blocks.0";
    Act k2 = linear(P, T.text, prep(b + ".attn2.to_k", {b + ".attn2.to_k"}));
    Act v2t = vt_proj(P, T.text, T.text_batch, 77, prep(b + ".attn2.to_v", {b + ".attn2.to_v"}));
    T.kv[b] = std::make_pair(k2, v2t);
  }
  flush_prep();
  I2IT_CUDA(cudaDeviceSynchronize());
}

Act Engine::build_unet(Plan& P, const Act& z, int text_batch, bool text_cached) {
  const std::string u = "unet";
  const int* ch = cfg.unet_channels;
  const int* heads = cfg.unet_heads;
  text_kv_ = nullptr;
  if (text_cached) {
    auto it = textkv_.find(text_batch);
    I2IT_CHECK(it != textkv_.end(), "text_emb == NULL but i2it_set_text has not been called for this text_batch since the last "
                                    "i2it_finalize_weights");
    text_kv_ = it->second.get();
  } else {
    // stage the text embedding: its projections are TMA operands, whose maps need a fixed base address
    text_ = alloc_act(P, text_batch, 1, 77, cfg.cross_dim);
    P.keep.push_back(text_.hold);
    uint16_t* tp = text_.p;
    const size_t bytes = static_cast<size_t>(text_batch) * 77 * cfg.cross_dim * 2;
    Plan* plan = &P;
    add_op(P, [=](cudaStream_t st) {
      cudaMemcpyAsync(tp, plan->io.text, bytes, cudaMemcpyDeviceToDevice, st);
    });
  }
  // torch.cat([h, skip], dim=1) without copies: every skip connection is produced straight into the upper channel slice of
  // the concat buffer its up-block resnet will read, and the running `h` into the lower slice.
  // Consumer q (pop order, 3 per up block) needs sC(q) channels of `h` in front of the skip.
  struct SkipSlot { Act cat, skip; int sC; };
  std::vector<SkipSlot> res;
  const int rch[4] = {ch[3], ch[2], ch[1], ch[0]};
  const int total_pushes = 12;                       // conv_in + 4 x 2 block outputs + 3 downsamplers
  int pushes = 0;
  auto make_slot = [&](int N, int H, int W, int skipC) {
    const int q = total_pushes - 1 - pushes++, i = q / 3, j = q % 3;
    SkipSlot t;
    t.sC = (j == 0) ? (i == 0 ? ch[3] : rch[i - 1]) : rch[i];
    t.cat = alloc_act(P, N, H, W, t.sC + skipC);
    t.skip = t.cat.slice(t.sC, skipC);
    return t;
  };
  auto push = [&](SkipSlot& t, const Act& produced) { t.skip = produced; res.push_back(t); };   // keeps the producer's GN partials
  auto h_target = [&]() { return res.back().cat.slice(0, res.back().sC); };                      // where the next `h` goes

  Act s;
  {
    SkipSlot t = make_slot(z.N, z.H, z.W, ch[0]);
    ConvOpts oc; oc.gn_out = true; oc.out = &t.skip;
    if (has(u + ".conv_in.conv_in_pretrained.weight"))
      s = conv(P, z, prep_twin(u + ".conv_in.conv_in_pretrained", u + ".conv_in.conv_in_curr", twin_r_), oc);
    else
      s = conv(P, z, prep(u + ".conv_in", {u + ".conv_in"}), oc);
    push(t, s);
  }
  for (int i = 0; i < 4; ++i) {
    const std::string blk = u + ".down_blocks." + std::to_string(i);
    for (int j = 0; j < 2; ++j) {
      // who consumes the output decides whether the producing GEMM takes GroupNorm statistics: the transformer's GroupNorm
      // (i < 3), the next resnet's norm1 (j == 0, or the mid block after the last down block) — not the downsampler conv
      SkipSlot t = make_slot(s.N, s.H, s.W, ch[i]);
      s = unet_resnet(P, blk + ".resnets." + std::to_string(j), s, true, i < 3 ? nullptr : &t.skip);
      if (i < 3) s = unet_xformer(P, blk + ".attentions." + std::to_string(j), s, heads[i], text_batch, j == 0, &t.skip);
      push(t, s);
    }
    if (i < 3) {
      SkipSlot t = make_slot(s.N, (s.H + 1) / 2, (s.W + 1) / 2, ch[i]);
      ConvOpts o; o.stride = 2; o.gn_out = true; o.out = &t.skip;
      s = conv(P, s, prep(blk + ".downsamplers.0.conv", {blk + ".downsamplers.0.conv"}), o);
      push(t, s);
    }
  }
  I2IT_CHECK(pushes == total_pushes, "unet: unexpected number of skip connections");
  s = unet_resnet(P, u + ".mid_block.resnets.0", s, true);
  s = unet_xformer(P, u + ".mid_block.attentions.0", s, heads[3], text_batch, true);
  {
    const Act tgt = h_target();
    s = unet_resnet(P, u + ".mid_block.resnets.1", s, false, &tgt);   // -> concat (GroupNorm over the concatenation)
  }
  mark(P, "unet_mid", s);
  for (int i = 0; i < 4; ++i) {
    const std::string blk = u + ".up_blocks." + std::to_string(i);
    const int hcount = heads[3 - i];
    for (int j = 0; j < 3; ++j) {
      SkipSlot t = res.back();
      res.pop_back();
      I2IT_CHECK(s.C == t.sC && s.p == t.cat.p && s.H == t.cat.H && s.W == t.cat.W, "unet: concat slot mismatch");
      const Act cat = t.cat;                                           // both halves were written in place
      t = SkipSlot();
      const bool last = (i == 3 && j == 2);                            // the very last block feeds conv_norm_out directly
      // the block's output is the next concat's `h` unless an upsampler (j == 2, i < 3) or conv_norm_out (last) follows
      Act tgt;
      if (j < 2) tgt = h_target();
      const Act* ov = j < 2 ? &tgt : nullptr;
      s = unet_resnet(P, blk + ".resnets." + std::to_string(j), cat, i > 0, i > 0 ? nullptr : ov);
      if (i > 0) s = unet_xformer(P, blk + ".attentions." + std::to_string(j), s, hcount, text_batch, last, ov);
    }
    if (i < 3) {
      // Upsample2D: 2x nearest, or — when the latent is not a multiple of 8 (UNet2DConditionModel.forward: forward_upsample_size)
      // — nearest to the spatial size of the next skip connection (e.g. 14 -> 27 columns for a 560x840 image)
      const SkipSlot& nxt = res.back();
      s = upsample_to(P, s, nxt.skip.H, nxt.skip.W);
      const Act tgt = h_target();
      ConvOpts oc; oc.out = &tgt;
      s = conv(P, s, prep(blk + ".upsamplers.0.conv", {blk + ".upsamplers.0.conv"}), oc);
    }
  }
  I2IT_CHECK(res.empty(), "unet: residual stack not consumed");
  (void)ch;
  s = group_norm(P, s, norm(u + ".conv_norm_out"), 1e-5f, true);
  s = conv(P, s, prep(u + ".conv_out", {u + ".conv_out"}), ConvOpts());
  text_ = Act();
  text_kv_ = nullptr;
  return s;
}

// ------------------------------------------------------------------------------------------ whole path
Plan* Engine::plan_for(int B, int H, int W, int direction, int text_batch, bool text_cached, int io_mode) {
  const std::vector<int> key{B, H, W, direction, text_batch, text_cached ? 1 : 0, io_mode};
  auto it = plans_.find(key);
  if (it != plans_.end()) return it->second.get();
  I2IT_CHECK(finalized_, "i2it_finalize_weights must be called before a forward");
  std::string vp = "vae.";
  if (cfg.model_kind == I2IT_CYCLEGAN && direction == I2IT_B2A) vp = "vae_b2a.";
  std::unique_ptr<Plan> up(new Plan());
  Plan& P = *up;
  P.key = key;
  // a build that throws must not leave engine members pointing into the dying plan's pool (text_ holds a pool block):
  // declared after `up`, so it runs before the plan is destroyed
  struct BuildGuard {
    Engine* e; bool ok = false;
    ~BuildGuard() { if (!ok) { e->text_ = Act(); e->text_kv_ = nullptr; } }
  } guard{this};
  std::vector<Act> skips;
  if (io_mode & IO_U8_OUT) {
    // allocated FIRST and held for the plan's lifetime: pool liveness follows build order, and the last conv writes here
    auto tmp = alloc_raw(P, static_cast<size_t>(B) * 3 * H * W * 2);
    P.keep.push_back(tmp);
    P.u8_out_tmp = tmp.get();
  }
  P.ranges.emplace_back(P.ops.size(), "vae_encode");
  Act z = build_vae_encoder(P, vp, B, H, W, skips, (io_mode & IO_U8_IN) != 0);
  P.ranges.emplace_back(P.ops.size(), "unet");
  Act pred = build_unet(P, z, text_batch, text_cached);
  mark(P, "model_pred", pred);
  P.ranges.emplace_back(P.ops.size(), "ddpm_step");
  Act dec_in = alloc_act(P, B, H / 8, W / 8, 8, 8, true);
  {
    // alpha_bar_999 of the scaled-linear schedule (fp32 cumprod, as diffusers computes it): 0.0046600951
    const float sa = 0.06826488673686981f, s1 = 0.9976672530174255f, inv_sf = 1.0f / cfg.scaling_factor;
    const long long HW = static_cast<long long>(H / 8) * (W / 8), total = HW * B;
    const uint16_t* zp = z.p;
    const uint16_t* pp = pred.p;
    uint16_t* dp = dec_in.p;
    const int ldp = pred.ld, dt = dtype;
    // the two wrappers call DDPMScheduler.step with different timestep shapes => different rounding (kernels.cuh)
    const int three_round = (cfg.model_kind == I2IT_CYCLEGAN) ? 1 : 0;
    Plan* plan = &P;
    P.keep.push_back(z.hold);
    P.keep.push_back(pred.hold);
    add_op(P, [=](cudaStream_t st) {
      DISPATCH_T(dt, (launch_k(ddpm_step_kernel<T>, dim3(ceil_div_i(total, 128)), dim3(128), 0, st, 0,
                         reinterpret_cast<const T*>(zp), reinterpret_cast<const T*>(pp), ldp, s1, sa, inv_sf,
                         reinterpret_cast<T*>(dp), reinterpret_cast<T*>(plan->io.out_latent), HW, total, three_round)));
    });
  }
  mark(P, "dec_in", dec_in);
  P.ranges.emplace_back(P.ops.size(), "vae_decode");
  build_vae_decoder(P, vp, dec_in, skips);
  if (io_mode & IO_U8_OUT) {
    // the last conv wrote NCHW into an internal buffer (forward() points io.out at it); convert to uint8 HWC for the caller
    const long long HW = static_cast<long long>(H) * W, total = HW * B;
    const int dt = dtype;
    Plan* plan = &P;
    add_op(P, [=](cudaStream_t st) {
      DISPATCH_T(dt, (launch_k(nchw_to_u8hwc_kernel<T>, dim3(ceil_div_i(total, 256)), dim3(256), 0, st, 0,
                         reinterpret_cast<const T*>(plan->io.out), reinterpret_cast<uint8_t*>(plan->io.out_u8), HW, total)));
    }, "unpack_u8", 0, 1.0 * total * (6 + 3));
  }
  flush_prep();                             // every weight of the plan: one fold/re-layout launch (+ the time-embedding GEMVs)
  I2IT_CUDA(cudaDeviceSynchronize());       // weight preparation ran on the default stream
  I2IT_CUDA(cudaGetLastError());
  Plan* raw_plan = up.get();
  plans_[key] = std::move(up);
  guard.ok = true;
  return raw_plan;
}

}  // namespace i2it
