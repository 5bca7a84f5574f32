/*
 * death_fog_oracle.h -- the death fog of Player.update, as the CPU reference the device's fog is checked against.
 *
 * tests/fog_oracle.py compiles oracle/nmmo_oracle.c with this file included just before player_update, and a call
 * `if (death_fog_update(e, row)) return;` at the start of its Resources.update part; every other line of the oracle is
 * the one all the other parity tests use.  With NC_DEATH_FOG = -1 the function does nothing.
 *
 * [UPSTREAM nmmo/entity/player.py Player.update], restated (the engine is not vendored).  It runs in players.update,
 * after the Entity.update / History.update part and before Resources.update; realm.tick = e->tick, the tick before the
 * step increments it (an onset of 0 = fog from the first step after a reset):
 *
 *   fog = config.PLAYER_DEATH_FOG                      # None = off
 *   if fog is not None and realm.tick >= fog:
 *       row, col = self.pos
 *       cent = config.MAP_BORDER + config.MAP_CENTER // 2
 *       dist = max(abs(row - cent), abs(col - cent))
 *       if dist > config.PLAYER_DEATH_FOG_FINAL_SIZE:                       # default 8
 *           time_dmg = config.PLAYER_DEATH_FOG_SPEED * (realm.tick - fog + 1)  # default 1
 *           dist_dmg = dist - config.MAP_CENTER // 2
 *           self.receive_damage(None, max(0, dist_dmg + time_dmg))
 *   if not self.alive:
 *       return                      # no Resources.update, no Skills.update this tick
 *   self.resources.update(); self.skills.update()
 *
 * receive_damage(None, dmg): damage_received += dmg (saturating at 32767 as in act_attack), damage = dmg (not clamped to
 * health), health = max(0, health - dmg).  A player it kills has no source to loot it: all of its items are unlisted
 * and destroyed at once, here, inside the id-ordered players.update loop (item_destroy also unlists); its gold stays
 * with the corpse.  No event, no kill credit; spawn immunity does not apply; NPCs are never touched (NPC.update has no
 * fog).  A player that reaches players.update is alive (the cull removes the others), so only the fog can kill it here.
 */

/* 1: the fog killed the player (its Resources / Skills update is skipped) */
static int death_fog_update(OEnv *e, int row) {
  int32_t *a = e->ent[row];
  const int32_t *c = e->cfg;
  if (c[NC_DEATH_FOG] < 0 || e->tick < c[NC_DEATH_FOG]) return 0;
  int cent = c[NC_MAP_BORDER] + c[NC_MAP_CENTER] / 2;
  int dist = imax(abs(a[EA_ROW] - cent), abs(a[EA_COL] - cent));
  if (dist <= c[NC_DEATH_FOG_FINAL_SIZE]) return 0;
  int time_dmg = c[NC_DEATH_FOG_SPEED] * (e->tick - c[NC_DEATH_FOG] + 1);
  int dmg = imax(0, dist - c[NC_MAP_CENTER] / 2 + time_dmg);
  a[EA_DMG_RECEIVED] = imin(32767, a[EA_DMG_RECEIVED] + dmg);
  a[EA_DAMAGE] = dmg;
  a[EA_HEALTH] = imax(0, a[EA_HEALTH] - dmg);
  if (a[EA_HEALTH] > 0) return 0;
  for (int i = 0; i < e->cap; i++) if (e->items[i].used && e->items[i].owner == a[EA_ID]) item_destroy(e, i);
  return 1;
}
