/* tbx_host.h -- host-side (no CUDA) half of the library: default configs, geometry tables, the JSON
 * codecs for config and state in the reference's schema, JSON-schema export, INTER_AREA tap tables.
 * Everything here runs once per pool / per intervention, never per frame.
 */
#ifndef TBX_HOST_H
#define TBX_HOST_H
#include "tbx_records.h"
#include "tbx_json.h"
#include <string>
#include <vector>

struct TbxBrkDirect; /* tbx_direct.h */
struct TbxSiDirect;
struct TbxAmiDirect;
struct TbxSpritePatch;

namespace tbx {

struct GameInfo {
  int id;
  const char *name;
  int width, height;
  int n_legal;
  int legal[18];
  int rec_words;
  int n_slots;
  int new_games_at_ctor; /* SURVEY App. A.2: fixture lineage */
};
const GameInfo *game_info(int game);
int game_from_name(const char *name); /* -1 if unknown */

/* one pool-level config, whichever game */
struct Config {
  int game;
  BrkCfg brk;
  SiCfg si;
  AmiCfg ami;
};
void default_config(int game, Config &c);
void brk_finish_cfg(BrkCfg &c); /* validates and fills the host-evaluated trig tables */
tbxjson::Value config_to_json(const Config &c);
void config_from_json(Config &c, const tbxjson::Value &v); /* throws std::runtime_error */

/* geometry tables */
void brk_default_table(const BrkCfg &c, BrkTable &t);
void brk_finish_table(BrkTable &t); /* derived fields (x1,y1, ints, bbox, masks, disjoint) from px..color,destructible */
void ami_default_table(const AmiCfg &c, AmiTable &t);
void ami_finish_table(AmiTable &t);

/* state records <-> JSON.  `table` is the geometry table the record refers to (to_json) or the table
 * the JSON describes (from_json; the caller interns it and sets rec.hdr.tbl). */
tbxjson::Value brk_state_to_json(const BrkRec &r, const BrkTable &t);
void brk_state_from_json(const tbxjson::Value &v, BrkRec &r, BrkTable &t);
tbxjson::Value si_state_to_json(const SiRec &r);
void si_state_from_json(const tbxjson::Value &v, SiRec &r);
tbxjson::Value ami_state_to_json(const AmiRec &r, const AmiTable &t);
void ami_state_from_json(const tbxjson::Value &v, AmiRec &r, AmiTable &t);

/* Toybox.query_state_json(query, args) (toybox/interventions/amidar.py:508-518): amidar tile_to_world /
 * world_to_tile; breakout bricks_remaining / count_channels / channels.  `rec` is the env's record, `brk` its
 * brick table (breakout only).  Throws on an unknown query. */
tbxjson::Value query_json(int game, const uint32_t *rec, const BrkTable *brk, const std::string &query, const tbxjson::Value &args);

tbxjson::Value schema_for_state(int game);
tbxjson::Value schema_for_config(int game);

/* cv2.resize(..., INTER_AREA) tap tables, general (non-integer scale) path
 * (baselines/baselines/common/atari_wrappers.py:243) */
typedef TbxResizeAxis ResizeAxis;
typedef TbxResizeTab ResizeTab;
void build_resize(int sw, int sh, int dw, int dh, ResizeTab &t); /* throws if the size pair is not on the general path */
/* repack for the fused kernel; returns false when the size pair exceeds its limits (the generic kernel handles those) */
bool build_area_plan(const ResizeTab &t, TbxAreaPlan &plan);

/* Static part of a game's frame: the leading draw-list slots that depend on the config only (Breakout: frame
 * walls; Space Invaders: ground line; Amidar: none) painted over the clear colour.  rgba: W*H pixels. */
int n_static_slots(int game);
/* base_id 0: static slots only.  base_id 1: plus the reference (new_game) look of the delta-rendered group --
 * Breakout: every brick of `brk_default` alive; Amidar: the config board's tiles (tbx_*_prim_delta). */
void build_base_frame(const Config &c, const BrkTable *brk_default, int base_id, uint32_t *rgba);
/* sets t.delta_ok for the config (same answer for identical tables, so interning is unaffected) */
void brk_mark_delta_ok(const Config &c, BrkTable &t);
/* gray bytes of an RGBA frame, and its INTER_AREA down-sample (same arithmetic as the kernels) */
void frame_to_gray(const uint32_t *rgba, int npix, uint8_t *gray);
void area_resize(const uint8_t *gray, const ResizeTab &t, uint8_t *out);
/* the TBX_DP_SLOTS x 10 digit patches of base frame `base_id` (gray) for one output size; out[slot * 10 + digit] */
void build_digit_patches(const Config &c, const BrkTable *brk_default, const ResizeTab &t, const TbxAreaPlan &plan, const uint8_t *base_gray,
                         TbxDigitPatch *out);
/* closed-form tables of the direct INTER_AREA kernel (tbx_direct.h) for the config's default brick table and one output
 * size; out.ok == 0 when the pair is outside its limits (irregular brick grid, output width not a multiple of 4 ...) */
void build_brk_direct(const Config &c, const BrkTable &t, const ResizeTab &rs, const TbxAreaPlan &plan, const uint8_t *base0_gray, TbxBrkDirect &out);
/* the Breakout direct kernel's shared-memory image (tbx_direct.h) for tables A (A.ok) and the kernel instantiated for tx x ty taps:
 * base1_out is the down-sample of base frame 1, patches1 its TBX_DP_SLOTS x 10 digit patches */
void build_brk_img(const TbxBrkDirect &A, const TbxAreaPlan &plan, int tx, int ty, const uint8_t *base1_out, const TbxDigitPatch *patches1, std::vector<uint8_t> &img);
/* Space Invaders: plain-background map and pre-resolved sprite patch tables of the direct kernel (tbx_direct.h) */
void build_si_direct(const Config &c, const ResizeTab &rs, const TbxAreaPlan &plan, const uint8_t *base0_gray, TbxSiDirect &out, std::vector<TbxSpritePatch> &patches);
void build_ami_direct(const Config &c, const ResizeTab &rs, const TbxAreaPlan &plan, TbxAmiDirect &out); /* Amidar: tile-look tables of the direct kernel */
int digit_slot0(int game);   /* first draw-list slot of the HUD digit fields */
int digit_slots(int game);   /* how many consecutive digit slots follow */

} /* namespace tbx */
#endif
