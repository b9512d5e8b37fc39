// Encoder dimensions derived from a VitkConfig and a batch size, with the checks that inference
// (api.cu) and training (api_train.cu) share.
#pragma once
#include "../../include/vitk.h"

#include "common.h"

namespace vitk {

struct Dims {
  int B, S, p, C, D, L, H, Mlp, prefix, P, N, Kp, hd, ncls;
  long long M, Mp;  // token rows, patch rows
};

inline int check_config(const VitkConfig* cfg, int batch, Dims* d) {
  VITK_REQUIRE(cfg != nullptr, "config is null");
  VITK_REQUIRE(batch > 0, "batch must be positive (got %d)", batch);
  VITK_REQUIRE(cfg->image_size > 0 && cfg->patch_size > 0 &&
                   cfg->image_size % cfg->patch_size == 0,
               "image_size %d must be a positive multiple of patch_size %d", cfg->image_size,
               cfg->patch_size);
  VITK_REQUIRE(cfg->embed_dim > 0 && cfg->num_heads > 0 && cfg->embed_dim % cfg->num_heads == 0,
               "embed_dim %d must be divisible by num_heads %d", cfg->embed_dim, cfg->num_heads);
  VITK_REQUIRE(cfg->n_prefix_tokens == 1 || cfg->n_prefix_tokens == 2,
               "n_prefix_tokens must be 1 (ViT) or 2 (DeiT)");
  VITK_REQUIRE(cfg->num_layers > 0 && cfg->mlp_dim > 0 && cfg->in_channels > 0, "bad layer sizes");
  VITK_REQUIRE(cfg->embed_dim % 8 == 0 && cfg->mlp_dim % 8 == 0,
               "embed_dim and mlp_dim must be multiples of 8");
  d->B = batch;
  d->S = cfg->image_size;
  d->p = cfg->patch_size;
  d->C = cfg->in_channels;
  d->D = cfg->embed_dim;
  d->L = cfg->num_layers;
  d->H = cfg->num_heads;
  d->Mlp = cfg->mlp_dim;
  d->prefix = cfg->n_prefix_tokens;
  const int gw = d->S / d->p;
  d->P = gw * gw;
  d->N = d->P + d->prefix;
  d->Kp = d->C * d->p * d->p;
  d->hd = d->D / d->H;
  d->ncls = cfg->n_classes;
  d->M = static_cast<long long>(batch) * d->N;
  d->Mp = static_cast<long long>(batch) * d->P;
  VITK_REQUIRE(d->M < (1ll << 31) / 4, "batch too large");
  return VITK_OK;
}

}  // namespace vitk
