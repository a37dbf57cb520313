"""Rule names and orders of the reference's data.yaml, restated as Python constants.

Orders are semantics: inventory / item-strip order (data.yaml:39-55, engine.py:230,238), achievement
order (data.yaml:80-102), action ids (data.yaml:1-18), material ids = index + 1 (engine.py:29-30).
The numeric rule tables themselves (collect / place / make) live in csrc/cr_update.h.
"""

ACTIONS = [
    'noop', 'move_left', 'move_right', 'move_up', 'move_down', 'do', 'sleep', 'place_stone',
    'place_table', 'place_furnace', 'place_plant', 'make_wood_pickaxe', 'make_stone_pickaxe',
    'make_iron_pickaxe', 'make_wood_sword', 'make_stone_sword', 'make_iron_sword']

MATERIALS = [
    'water', 'grass', 'stone', 'path', 'sand', 'tree', 'lava', 'coal', 'iron', 'diamond', 'table',
    'furnace']

ITEMS = [
    'health', 'food', 'drink', 'energy', 'sapling', 'wood', 'stone', 'coal', 'iron', 'diamond',
    'wood_pickaxe', 'stone_pickaxe', 'iron_pickaxe', 'wood_sword', 'stone_sword', 'iron_sword']

ACHIEVEMENTS = [
    'collect_coal', 'collect_diamond', 'collect_drink', 'collect_iron', 'collect_sapling',
    'collect_stone', 'collect_wood', 'defeat_skeleton', 'defeat_zombie', 'eat_cow', 'eat_plant',
    'make_iron_pickaxe', 'make_iron_sword', 'make_stone_pickaxe', 'make_stone_sword',
    'make_wood_pickaxe', 'make_wood_sword', 'place_furnace', 'place_plant', 'place_stone',
    'place_table', 'wake_up']

# Sprite order of the object atlas (csrc/cr_common.h ObjTex).
OBJECT_SPRITES = [
    'player-left', 'player-right', 'player-up', 'player-down', 'player-sleep', 'cow', 'zombie',
    'skeleton', 'arrow-left', 'arrow-right', 'arrow-up', 'arrow-down', 'plant', 'plant-ripe']

# Semantic-view ids (engine.py:253-258 with env.py:47-49): materials 1..12, then these.
SEMANTIC_OBJECTS = ['player', 'cow', 'zombie', 'skeleton', 'arrow', 'plant']  # ids 13..18

# csrc/cr_common.h PState columns.
PSTATE = ['hunger2', 'thirst2', 'fatigue', 'recover2', 'sleeping', 'player_last_health',
          'env_last_health', 'unlocked', 'n_slots', 'step', 'episode', 'world_seed', 'player_x',
          'player_y', 'error', 'episode_length']

# The numeric rule tables (data.yaml:34-78), restated for documentation and for the tests that (a) diff
# them against the reference's data.yaml (tests/golden/data_yaml.json) and (b) probe the device code
# (csrc/cr_update.h player_do_material / player_place / player_make, csrc/cr_worldgen.h wg_fresh_player)
# with them, entry by entry (tests/test_rules_table.py).
WALKABLE = ['grass', 'sand', 'path']
ITEM_MAX = 9
ITEM_INITIAL = {'health': 9, 'food': 9, 'drink': 9, 'energy': 9}  # everything else 0
COLLECT = {  # material: (required tool or None, received item, material left behind, probability)
    'tree': (None, 'wood', 'grass', 1.0), 'stone': ('wood_pickaxe', 'stone', 'path', 1.0),
    'coal': ('wood_pickaxe', 'coal', 'path', 1.0), 'iron': ('stone_pickaxe', 'iron', 'path', 1.0),
    'diamond': ('iron_pickaxe', 'diamond', 'path', 1.0), 'water': (None, 'drink', 'water', 1.0),
    'grass': (None, 'sapling', 'grass', 0.1)}
PLACE = {  # name: (item used, amount, materials it may replace, 'material' | 'object')
    'stone': ('stone', 1, ['grass', 'sand', 'path', 'water', 'lava'], 'material'),
    'table': ('wood', 2, ['grass', 'sand', 'path'], 'material'),
    'furnace': ('stone', 4, ['grass', 'sand', 'path'], 'material'),
    'plant': ('sapling', 1, ['grass'], 'object')}
MAKE = {  # name: (items used, materials needed nearby)
    'wood_pickaxe': ({'wood': 1}, ['table']), 'stone_pickaxe': ({'wood': 1, 'stone': 1}, ['table']),
    'iron_pickaxe': ({'wood': 1, 'coal': 1, 'iron': 1}, ['table', 'furnace']),
    'wood_sword': ({'wood': 1}, ['table']), 'stone_sword': ({'wood': 1, 'stone': 1}, ['table']),
    'iron_sword': ({'wood': 1, 'coal': 1, 'iron': 1}, ['table', 'furnace'])}
